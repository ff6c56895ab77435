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


def _dims(adj, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh):
    if x.dim() != 4:
        raise RuntimeError(f"attr_matrix must be [B, T, S, F_in], got {tuple(x.shape)}")
    B, T, S, F_in = x.shape
    if adj.shape != (S, S):
        raise RuntimeError(f"adj_matrix must be [{S}, {S}], got {tuple(adj.shape)}")
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
    return B, T, S, F_in, F_hid, F_out, H


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
    lib = _lib.load()
    x = _require_cuda_f32("attr_matrix", x)
    dev = x.device
    adj, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh = (
        _require_cuda_f32(n, t, dev)
        for n, t in (
            ("adj_matrix", adj), ("conv1.weight", w1), ("conv1.bias", b1), ("conv2.weight", w2),
            ("conv2.bias", b2), ("gru.weight_ih_l0", w_ih), ("gru.weight_hh_l0", w_hh),
            ("gru.bias_ih_l0", b_ih), ("gru.bias_hh_l0", b_hh),
        )
    )
    B, T, S, F_in, F_hid, F_out, H = _dims(adj, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh)
    out = torch.empty((B, T, H), dtype=torch.float32, device=dev)
    if B == 0 or T == 0:
        return out
    # 0 bytes: the shape is rejected, and the call below returns the library's code and reason without launching
    nbytes = lib.wg_gcn_gru_workspace_bytes(B, T, S, F_in, F_hid, F_out, H, chunk, flags)
    ws = _workspace(dev, nbytes)
    stream = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(
        lib.wg_gcn_gru_forward_f32(
            adj.data_ptr(), x.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
            w_ih.data_ptr(), w_hh.data_ptr(), b_ih.data_ptr(), b_hh.data_ptr(), out.data_ptr(),
            B, T, S, F_in, F_hid, F_out, H, chunk, flags, ws.data_ptr(), ws.numel(), dev.index or 0, stream,
        )
    )
    return out


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
    lib = _lib.load()
    x = _require_cuda_f32("attr_matrix", x)
    dev = x.device
    w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, vals = (
        _require_cuda_f32(n, t, dev)
        for n, t in (
            ("conv1.weight", w1), ("conv1.bias", b1), ("conv2.weight", w2), ("conv2.bias", b2),
            ("gru.weight_ih_l0", w_ih), ("gru.weight_hh_l0", w_hh), ("gru.bias_ih_l0", b_ih),
            ("gru.bias_hh_l0", b_hh), ("adjacency values", vals),
        )
    )
    if x.dim() != 4:
        raise RuntimeError(f"attr_matrix must be [B, T, S, F_in], got {tuple(x.shape)}")
    S = x.shape[2]
    for n, t in (("rowptr", rowptr), ("colidx", colidx)):
        if not t.is_cuda or t.dtype != torch.int32 or t.device != dev:
            raise RuntimeError(f"windgnn_b200: {n} must be a CUDA int32 tensor on {dev}")
    rowptr, colidx = rowptr.contiguous(), colidx.contiguous()
    if rowptr.numel() != S + 1 or colidx.numel() != vals.numel():
        raise RuntimeError("CSR arrays do not match the number of stations")
    adj_shape = torch.empty((S, S), device="meta")
    B, T, S, F_in, F_hid, F_out, H = _dims(adj_shape, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh)
    out = torch.empty((B, T, H), dtype=torch.float32, device=dev)
    if B == 0 or T == 0:
        return out
    nbytes = lib.wg_gcn_gru_csr_workspace_bytes(B, T, S, F_in, F_hid, F_out, H, chunk, flags)  # 0: see gcn_gru_forward
    ws = _workspace(dev, nbytes)
    stream = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(
        lib.wg_gcn_gru_forward_csr_f32(
            rowptr.data_ptr(), colidx.data_ptr(), vals.data_ptr(), x.data_ptr(), w1.data_ptr(), b1.data_ptr(),
            w2.data_ptr(), b2.data_ptr(), w_ih.data_ptr(), w_hh.data_ptr(), b_ih.data_ptr(), b_hh.data_ptr(),
            out.data_ptr(), B, T, S, F_in, F_hid, F_out, H, chunk, flags, ws.data_ptr(), ws.numel(), dev.index or 0,
            stream,
        )
    )
    return out


@gcn_gru_forward_csr.register_fake
def _(rowptr, colidx, vals, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, chunk=0, flags=0):
    return x.new_empty((x.shape[0], x.shape[1], w_hh.shape[1]))


def _forecast_starts(starts: torch.Tensor) -> torch.Tensor:
    """The windows' first table rows as the contiguous HOST int64 array the library reads."""
    if not isinstance(starts, torch.Tensor) or starts.dtype != torch.int64 or starts.dim() != 1:
        raise RuntimeError("starts must be a 1-D int64 tensor")
    return starts.cpu().contiguous()


def _forecast_dims(adj, table, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh):
    if table.dim() != 3:
        raise RuntimeError(f"table must be [Ttot, S, F_in], got {tuple(table.shape)}")
    _, Ttot, S, F_in, F_hid, F_out, H = _dims(adj, table.unsqueeze(0), w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh)
    return Ttot, S, F_in, F_hid, F_out, H


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
    lib = _lib.load()
    table = _require_cuda_f32("table", table)
    dev = table.device
    adj, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh = (
        _require_cuda_f32(n, t, dev)
        for n, t in (
            ("adj_matrix", adj), ("conv1.weight", w1), ("conv1.bias", b1), ("conv2.weight", w2),
            ("conv2.bias", b2), ("gru.weight_ih_l0", w_ih), ("gru.weight_hh_l0", w_hh),
            ("gru.bias_ih_l0", b_ih), ("gru.bias_hh_l0", b_hh),
        )
    )
    Ttot, S, F_in, F_hid, F_out, H = _forecast_dims(adj, table, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh)
    starts = _forecast_starts(starts)
    N = starts.numel()
    out = torch.empty((N, H), dtype=torch.float32, device=dev)
    # 0 bytes: the shape is rejected, and the call below returns the library's code and reason without launching
    nbytes = lib.wg_gcn_gru_forecast_workspace_bytes(N, Ttot, seq_length, S, F_in, F_hid, F_out, H, chunk, flags)
    ws = _workspace(dev, nbytes, "forecast")
    stream = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(
        lib.wg_gcn_gru_forecast_f32(
            adj.data_ptr(), table.data_ptr(), starts.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
            b2.data_ptr(), w_ih.data_ptr(), w_hh.data_ptr(), b_ih.data_ptr(), b_hh.data_ptr(), out.data_ptr(),
            N, Ttot, seq_length, S, F_in, F_hid, F_out, H, chunk, flags, ws.data_ptr(), ws.numel(), dev.index or 0,
            stream,
        )
    )
    return out


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
    lib = _lib.load()
    table = _require_cuda_f32("table", table)
    dev = table.device
    w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, vals = (
        _require_cuda_f32(n, t, dev)
        for n, t in (
            ("conv1.weight", w1), ("conv1.bias", b1), ("conv2.weight", w2), ("conv2.bias", b2),
            ("gru.weight_ih_l0", w_ih), ("gru.weight_hh_l0", w_hh), ("gru.bias_ih_l0", b_ih),
            ("gru.bias_hh_l0", b_hh), ("adjacency values", vals),
        )
    )
    if table.dim() != 3:
        raise RuntimeError(f"table must be [Ttot, S, F_in], got {tuple(table.shape)}")
    S = table.shape[1]
    for n, t in (("rowptr", rowptr), ("colidx", colidx)):
        if not t.is_cuda or t.dtype != torch.int32 or t.device != dev:
            raise RuntimeError(f"windgnn_b200: {n} must be a CUDA int32 tensor on {dev}")
    rowptr, colidx = rowptr.contiguous(), colidx.contiguous()
    if rowptr.numel() != S + 1 or colidx.numel() != vals.numel():
        raise RuntimeError("CSR arrays do not match the number of stations")
    adj_shape = torch.empty((S, S), device="meta")
    Ttot, S, F_in, F_hid, F_out, H = _forecast_dims(adj_shape, table, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh)
    starts = _forecast_starts(starts)
    N = starts.numel()
    out = torch.empty((N, H), dtype=torch.float32, device=dev)
    nbytes = lib.wg_gcn_gru_forecast_csr_workspace_bytes(N, Ttot, seq_length, S, F_in, F_hid, F_out, H, chunk,
                                                         flags)  # 0: see gcn_gru_forecast
    ws = _workspace(dev, nbytes, "forecast")
    stream = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(
        lib.wg_gcn_gru_forecast_csr_f32(
            rowptr.data_ptr(), colidx.data_ptr(), vals.data_ptr(), table.data_ptr(), starts.data_ptr(),
            w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), w_ih.data_ptr(), w_hh.data_ptr(),
            b_ih.data_ptr(), b_hh.data_ptr(), out.data_ptr(), N, Ttot, seq_length, S, F_in, F_hid, F_out, H, chunk,
            flags, ws.data_ptr(), ws.numel(), dev.index or 0, stream,
        )
    )
    return out


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
    ``out_host`` is complete.  ``params`` = the 8 tensors in state_dict order, on the GPU.

    ``last_step_range=(wind_min, wind_max)``: only the last timestep of every window, de-normalised
    (what the reference's evaluation reads, main.py:103,116), comes back: ``out_host`` is ``[B, H]``."""
    lib = _lib.load()
    if x_host.is_cuda or x_host.dtype != torch.float32 or not x_host.is_contiguous():
        raise RuntimeError("x_host must be a contiguous float32 CPU tensor")
    adj = _require_cuda_f32("adj_matrix", adj)
    dev = adj.device if device is None else torch.device(device)
    w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh = (_require_cuda_f32(f"param{i}", t, dev) for i, t in enumerate(params))
    B, T, S, F_in, F_hid, F_out, H = _dims(adj, x_host, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh)
    shape = (B, H) if last_step_range is not None else (B, T, H)
    if out_host is None:
        out_host = torch.empty(shape, dtype=torch.float32, pin_memory=True)
    if out_host.is_cuda or out_host.dtype != torch.float32 or not out_host.is_contiguous() or out_host.shape != shape:
        raise RuntimeError(f"out_host must be a contiguous float32 CPU tensor {list(shape)}")
    if B == 0:
        return out_host
    nbytes = lib.wg_gcn_gru_host_workspace_bytes(B, T, S, F_in, F_hid, F_out, H, chunk, flags)  # 0: see gcn_gru_forward
    ws = _workspace(dev, nbytes, "host")
    torch.cuda.current_stream(dev).synchronize()  # parameters / adj may have been produced on it
    ptrs = (adj.data_ptr(), x_host.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
            w_ih.data_ptr(), w_hh.data_ptr(), b_ih.data_ptr(), b_hh.data_ptr(), out_host.data_ptr())
    if last_step_range is None:
        _lib.check(lib.wg_gcn_gru_forward_host_f32(*ptrs, B, T, S, F_in, F_hid, F_out, H, chunk, flags, ws.data_ptr(),
                                                   ws.numel(), dev.index or 0))
    else:
        _lib.check(lib.wg_gcn_gru_predict_host_f32(*ptrs, B, T, S, F_in, F_hid, F_out, H, chunk, flags,
                                                   float(last_step_range[0]), float(last_step_range[1]),
                                                   ws.data_ptr(), ws.numel(), dev.index or 0))
    return out_host
