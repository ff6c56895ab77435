"""torch custom ops over the C-ABI (CUDA only — there is no CPU implementation).

``windgnn::gcn_gru_forward``  the fused forward of ``GCN_GRU`` (reference:
                              src/step6_gcn_gru_combined_model.py:13-27)
``windgnn::gcn_gru_forecast``  the last hidden state of windows over one table, GCN and projection once per
                              table row (``GCN_GRU.forecast``)
``windgnn::gcn_layer``        one ``GraphConvLayer`` (reference: src/step5_gcn_layer_model.py:13-23)

PyTorch is the plumbing here: it owns device memory (inputs, output, the cached workspace)
and supplies the current stream; all arithmetic happens in ``libwindgnn_b200.so``.
"""

from __future__ import annotations

import threading
from typing import Dict, Tuple

import torch

from . import _lib

_WORKSPACES: Dict[Tuple[int, int, str], torch.Tensor] = {}
_WS_LOCK = threading.Lock()

# the GCN_GRU parameters in state_dict order, the order every entry point takes them in
PARAM_NAMES = (
    "conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias",
    "gru.weight_ih_l0", "gru.weight_hh_l0", "gru.bias_ih_l0", "gru.bias_hh_l0",
)


def _workspace(device: torch.device, nbytes: int, tag: str = "fwd") -> torch.Tensor:
    """Scratch per (device, CUDA stream, tag), grown on demand and reused.  The library calls are
    stream-ordered and keep no pointer after they return, so calls on ONE stream may share a buffer;
    calls on different streams (or from different threads, which have different current streams or
    serialise on the lock while looking the buffer up) get different buffers."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    key = (idx, torch.cuda.current_stream(device).cuda_stream, tag)
    with _WS_LOCK:
        ws = _WORKSPACES.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
            _WORKSPACES[key] = ws
    return ws


def release_workspaces() -> None:
    _WORKSPACES.clear()


def _require_cuda_f32(name: str, t: torch.Tensor, device=None) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(
            f"windgnn_b200: {name} is on {t.device}; the fused path is CUDA-only (no CPU fallback)"
        )
    if t.dtype != torch.float32:
        raise RuntimeError(f"windgnn_b200: {name} must be float32, got {t.dtype}")
    if device is not None and t.device != device:
        raise RuntimeError(f"windgnn_b200: {name} is on {t.device}, expected {device}")
    return t.contiguous()


def _params(params, device: torch.device) -> list:
    """The eight parameters (``PARAM_NAMES`` order), checked to be float32 on ``device``, contiguous."""
    return [_require_cuda_f32(n, p, device) for n, p in zip(PARAM_NAMES, params, strict=True)]


def _param_dims(S: int, F_in: int, params) -> Tuple[int, int, int]:
    """``(F_hid, F_out, H)`` of the eight parameters, checked against ``S`` stations of ``F_in`` features."""
    w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh = params
    if w1.dim() != 2 or w1.shape[0] != F_in:
        raise RuntimeError(f"conv1.weight must be [{F_in}, F_hid], got {tuple(w1.shape)}")
    F_hid = w1.shape[1]
    if b1.shape != (F_hid,) or w2.dim() != 2 or w2.shape[0] != F_hid:
        raise RuntimeError("conv1.bias / conv2.weight do not match conv1.weight")
    F_out = w2.shape[1]
    if b2.shape != (F_out,):
        raise RuntimeError("conv2.bias does not match conv2.weight")
    if w_hh.dim() != 2 or w_hh.shape[0] != 3 * w_hh.shape[1]:
        raise RuntimeError(f"gru.weight_hh_l0 must be [3H, H], got {tuple(w_hh.shape)}")
    H = w_hh.shape[1]
    if w_ih.shape != (3 * H, S * F_out):
        # the reference fails in view()/GRU with a RuntimeError for the same mismatch (step6:20,23)
        raise RuntimeError(
            f"gru.weight_ih_l0 is {tuple(w_ih.shape)} but the flattened GCN output has {S * F_out} "
            f"features and H = {H}"
        )
    if b_ih.shape != (3 * H,) or b_hh.shape != (3 * H,):
        raise RuntimeError("gru biases must be [3H]")
    return F_hid, F_out, H


def _graph(graph, S: int, device: torch.device) -> tuple:
    """The adjacency as the library takes it, checked for ``S`` stations on ``device``: a dense fp32 ``adj [S, S]``
    gives ``(adj,)``; CSR ``(rowptr, colidx, vals)`` (int32 ``[S+1]``, int32 ``[nnz]``, fp32 ``[nnz]``) gives the
    same three.  The tensors come back contiguous."""
    if isinstance(graph, torch.Tensor):
        adj = _require_cuda_f32("adj_matrix", graph, device)
        if adj.shape != (S, S):
            raise RuntimeError(f"adj_matrix must be [{S}, {S}], got {tuple(adj.shape)}")
        return (adj,)
    rowptr, colidx, vals = graph
    vals = _require_cuda_f32("adjacency values", vals, device)
    for n, t in (("rowptr", rowptr), ("colidx", colidx)):
        if not t.is_cuda or t.dtype != torch.int32 or t.device != device:
            raise RuntimeError(f"windgnn_b200: {n} must be a CUDA int32 tensor on {device}")
    rowptr, colidx = rowptr.contiguous(), colidx.contiguous()
    if rowptr.numel() != S + 1 or colidx.numel() != vals.numel():
        raise RuntimeError("CSR arrays do not match the number of stations")
    return rowptr, colidx, vals


def _attr_shape(x: torch.Tensor) -> torch.Size:
    if x.dim() != 4:
        raise RuntimeError(f"attr_matrix must be [B, T, S, F_in], got {tuple(x.shape)}")
    return x.shape


def _run(query: str, entry: str, tensors, dims, device: torch.device, tag: str, extra=(), host: bool = False):
    """``entry(*pointers of tensors, *dims, *extra, workspace, its bytes, device index, current stream)`` with the
    cached workspace ``query(*dims)`` asks for; a non-zero status raises ``_lib.WindGNNError``.  A query returns 0
    bytes for a shape its entry point rejects, and the entry point then returns the library's code and reason
    without launching anything.  ``host``: the host-buffer entry points, which take no stream and run on streams of
    their own."""
    lib = _lib.load()
    ws = _workspace(device, getattr(lib, query)(*dims), tag)
    stream = torch.cuda.current_stream(device)
    args = (*(t.data_ptr() for t in tensors), *dims, *extra, ws.data_ptr(), ws.numel(), device.index or 0)
    if host:
        stream.synchronize()  # parameters / adj may have been produced on it
        _lib.check(getattr(lib, entry)(*args))
    else:
        _lib.check(getattr(lib, entry)(*args, stream.cuda_stream))


def _forward(query: str, entry: str, graph, x, params, chunk: int, flags: int) -> torch.Tensor:
    x = _require_cuda_f32("attr_matrix", x)
    dev = x.device
    B, T, S, F_in = _attr_shape(x)
    graph = _graph(graph, S, dev)
    params = _params(params, dev)
    F_hid, F_out, H = _param_dims(S, F_in, params)
    out = torch.empty((B, T, H), dtype=torch.float32, device=dev)
    if B == 0 or T == 0:
        return out
    _run(query, entry, (*graph, x, *params, out), (B, T, S, F_in, F_hid, F_out, H, chunk, flags), dev, "fwd")
    return out


def _forecast_starts(starts) -> torch.Tensor:
    """The windows' first table rows as the contiguous HOST int64 array the library reads (and range-checks)."""
    if not isinstance(starts, torch.Tensor) or starts.dtype != torch.int64 or starts.dim() != 1:
        raise RuntimeError("starts must be a 1-D int64 tensor")
    return starts.cpu().contiguous()


def _table_shape(table: torch.Tensor) -> torch.Size:
    if table.dim() != 3:
        raise RuntimeError(f"table must be [Ttot, S, F_in], got {tuple(table.shape)}")
    return table.shape


def _forecast(query: str, entry: str, graph, table, starts, params, seq_length: int, chunk: int,
              flags: int) -> torch.Tensor:
    table = _require_cuda_f32("table", table)
    dev = table.device
    Ttot, S, F_in = _table_shape(table)
    graph = _graph(graph, S, dev)
    params = _params(params, dev)
    F_hid, F_out, H = _param_dims(S, F_in, params)
    starts = _forecast_starts(starts)
    N = starts.numel()
    out = torch.empty((N, H), dtype=torch.float32, device=dev)
    # N == 0 goes to the library too: it still rejects a bad seq_length / Ttot
    _run(query, entry, (*graph, table, starts, *params, out),
         (N, Ttot, seq_length, S, F_in, F_hid, F_out, H, chunk, flags), dev, "forecast")
    return out


@torch.library.custom_op("windgnn::gcn_gru_forward", mutates_args=())
def gcn_gru_forward(
    adj: torch.Tensor,
    x: torch.Tensor,
    w1: torch.Tensor,
    b1: torch.Tensor,
    w2: torch.Tensor,
    b2: torch.Tensor,
    w_ih: torch.Tensor,
    w_hh: torch.Tensor,
    b_ih: torch.Tensor,
    b_hh: torch.Tensor,
    chunk: int = 0,
    flags: int = 0,
) -> torch.Tensor:
    """``x [B,T,S,F_in] -> [B,T,H]`` (every GRU hidden state), fused on the GPU.
    ``flags``: 0 = FP32 FMA everywhere, ``_lib.FLAG_TENSOR_CORES`` = 3xTF32 tcgen05 input projection."""
    return _forward("wg_gcn_gru_workspace_bytes", "wg_gcn_gru_forward_f32", adj, x,
                    (w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh), chunk, flags)


@gcn_gru_forward.register_fake
def _(adj, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, chunk=0, flags=0):
    return x.new_empty((x.shape[0], x.shape[1], w_hh.shape[1]))


@torch.library.custom_op("windgnn::gcn_gru_forward_csr", mutates_args=())
def gcn_gru_forward_csr(
    rowptr: torch.Tensor,
    colidx: torch.Tensor,
    vals: torch.Tensor,
    x: torch.Tensor,
    w1: torch.Tensor,
    b1: torch.Tensor,
    w2: torch.Tensor,
    b2: torch.Tensor,
    w_ih: torch.Tensor,
    w_hh: torch.Tensor,
    b_ih: torch.Tensor,
    b_hh: torch.Tensor,
    chunk: int = 0,
    flags: int = 0,
) -> torch.Tensor:
    """The same forward with the adjacency in CSR form (int32 ``rowptr [S+1]``, ``colidx [nnz]``,
    fp32 ``vals [nnz]``): the large-sparse-graph path (thousands of stations, wide GCN hidden layer).
    ``flags``: as for ``gcn_gru_forward`` (the tensor path serves the projection and the recurrence)."""
    return _forward("wg_gcn_gru_csr_workspace_bytes", "wg_gcn_gru_forward_csr_f32", (rowptr, colidx, vals), x,
                    (w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh), chunk, flags)


@gcn_gru_forward_csr.register_fake
def _(rowptr, colidx, vals, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, chunk=0, flags=0):
    return x.new_empty((x.shape[0], x.shape[1], w_hh.shape[1]))


@torch.library.custom_op("windgnn::gcn_gru_forecast", mutates_args=())
def gcn_gru_forecast(
    adj: torch.Tensor,
    table: torch.Tensor,
    starts: torch.Tensor,
    w1: torch.Tensor,
    b1: torch.Tensor,
    w2: torch.Tensor,
    b2: torch.Tensor,
    w_ih: torch.Tensor,
    w_hh: torch.Tensor,
    b_ih: torch.Tensor,
    b_hh: torch.Tensor,
    seq_length: int,
    chunk: int = 0,
    flags: int = 0,
) -> torch.Tensor:
    """Rolling forecasts: ``table [Ttot, S, F_in]`` and int64 ``starts [N]`` -> ``[N, H]``, row ``n`` the last
    hidden state of the window ``table[starts[n] : starts[n] + seq_length]``, bit-identical to
    ``gcn_gru_forward(window)[:, -1]`` with the same ``chunk`` and ``flags``.  GCN and input projection run once
    per table row.  ``starts`` may live on either device (the library reads it from the host)."""
    return _forecast("wg_gcn_gru_forecast_workspace_bytes", "wg_gcn_gru_forecast_f32", adj, table, starts,
                     (w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh), seq_length, chunk, flags)


@gcn_gru_forecast.register_fake
def _(adj, table, starts, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, seq_length, chunk=0, flags=0):
    return table.new_empty((starts.shape[0], w_hh.shape[1]))


@torch.library.custom_op("windgnn::gcn_gru_forecast_csr", mutates_args=())
def gcn_gru_forecast_csr(
    rowptr: torch.Tensor,
    colidx: torch.Tensor,
    vals: torch.Tensor,
    table: torch.Tensor,
    starts: torch.Tensor,
    w1: torch.Tensor,
    b1: torch.Tensor,
    w2: torch.Tensor,
    b2: torch.Tensor,
    w_ih: torch.Tensor,
    w_hh: torch.Tensor,
    b_ih: torch.Tensor,
    b_hh: torch.Tensor,
    seq_length: int,
    chunk: int = 0,
    flags: int = 0,
) -> torch.Tensor:
    """``gcn_gru_forecast`` with the adjacency in CSR form (as for ``gcn_gru_forward_csr``); bit-identical to
    ``gcn_gru_forward_csr(window)[:, -1]``."""
    return _forecast("wg_gcn_gru_forecast_csr_workspace_bytes", "wg_gcn_gru_forecast_csr_f32",
                     (rowptr, colidx, vals), table, starts, (w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh), seq_length,
                     chunk, flags)


@gcn_gru_forecast_csr.register_fake
def _(rowptr, colidx, vals, table, starts, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, seq_length, chunk=0, flags=0):
    return table.new_empty((starts.shape[0], w_hh.shape[1]))


def dense_to_csr(adj: torch.Tensor):
    """(rowptr int32 [S+1], colidx int32 [nnz], vals fp32 [nnz]) of a dense CUDA adjacency, columns
    ascending within a row.  Index plumbing only (torch); the arithmetic stays in the library."""
    adj = _require_cuda_f32("adj_matrix", adj)
    csr = adj.to_sparse_csr()
    return (csr.crow_indices().to(torch.int32).contiguous(), csr.col_indices().to(torch.int32).contiguous(),
            csr.values().contiguous())


@torch.library.custom_op("windgnn::gcn_layer", mutates_args=())
def gcn_layer(adj: torch.Tensor, attr: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """``relu((adj @ attr) @ weight + bias)`` for ``attr [..., S, F_in]``."""
    lib = _lib.load()
    attr = _require_cuda_f32("attr_matrix", attr)
    dev = attr.device
    adj = _require_cuda_f32("adj_matrix", adj, dev)
    weight = _require_cuda_f32("weight", weight, dev)
    bias = _require_cuda_f32("bias", bias, dev)
    if attr.dim() < 2:
        raise RuntimeError("attr_matrix must be [..., S, F_in]")
    S, F_in = attr.shape[-2], attr.shape[-1]
    if adj.shape != (S, S) or weight.dim() != 2 or weight.shape[0] != F_in or bias.shape != (weight.shape[1],):
        raise RuntimeError("gcn_layer: inconsistent shapes")
    F_out = weight.shape[1]
    R = attr.numel() // (S * F_in) if attr.numel() else 0
    out = torch.empty((*attr.shape[:-1], F_out), dtype=torch.float32, device=dev)
    if R == 0:
        return out
    stream = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(
        lib.wg_gcn_layer_f32(
            adj.data_ptr(), attr.data_ptr(), weight.data_ptr(), bias.data_ptr(), out.data_ptr(),
            R, S, F_in, F_out, dev.index or 0, stream,
        )
    )
    return out


@gcn_layer.register_fake
def _(adj, attr, weight, bias):
    return attr.new_empty((*attr.shape[:-1], weight.shape[1]))


def gcn_gru_forward_host(adj, x_host, params, out_host=None, chunk: int = 0, device=None, flags: int = 0,
                         last_step_range=None):
    """End-to-end variant: ``x_host`` / ``out_host`` are HOST tensors (pin them for full
    copy/compute overlap); the batch is streamed through the GPU in chunks.  Blocks until
    ``out_host`` is complete.  ``params`` = the 8 tensors in state_dict order, on the GPU (``device``, by default
    the device of ``adj``).

    ``last_step_range=(wind_min, wind_max)``: only the last timestep of every window, de-normalised
    (what the reference's evaluation reads, main.py:103,116), comes back: ``out_host`` is ``[B, H]``."""
    if x_host.is_cuda or x_host.dtype != torch.float32 or not x_host.is_contiguous():
        raise RuntimeError("x_host must be a contiguous float32 CPU tensor")
    B, T, S, F_in = _attr_shape(x_host)
    if not isinstance(adj, torch.Tensor):  # the host entry points take the dense adjacency only
        raise TypeError("adj_matrix must be a torch.Tensor")
    dev = adj.device if device is None else torch.device(device)
    (adj,) = _graph(adj, S, dev)
    params = _params(params, dev)
    F_hid, F_out, H = _param_dims(S, F_in, params)
    shape = (B, H) if last_step_range is not None else (B, T, H)
    if out_host is None:
        out_host = torch.empty(shape, dtype=torch.float32, pin_memory=True)
    if out_host.is_cuda or out_host.dtype != torch.float32 or not out_host.is_contiguous() or out_host.shape != shape:
        raise RuntimeError(f"out_host must be a contiguous float32 CPU tensor {list(shape)}")
    if B == 0:
        return out_host
    tensors, dims = (adj, x_host, *params, out_host), (B, T, S, F_in, F_hid, F_out, H, chunk, flags)
    if last_step_range is None:
        _run("wg_gcn_gru_host_workspace_bytes", "wg_gcn_gru_forward_host_f32", tensors, dims, dev, "host", host=True)
    else:
        _run("wg_gcn_gru_host_workspace_bytes", "wg_gcn_gru_predict_host_f32", tensors, dims, dev, "host",
             extra=(float(last_step_range[0]), float(last_step_range[1])), host=True)
    return out_host
