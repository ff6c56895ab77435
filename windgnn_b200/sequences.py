"""step4 window extraction and the caller's de-normalisation, on the GPU.

Reference: ``__create_sequences`` (src/step4_sequence_preparer.py:7-27) and the de-normalise /
last-timestep selection of src/main.py:103,116,131,146.  The device works on the numeric block
of the reference's pivoted ``[time, station, 15]`` table: ``table[..., f]`` is column ``f + 2``
(``x = data[..., 2:15]``, step4:13), the label column 13 is feature 11.
"""

from __future__ import annotations

import torch

from . import _lib

SEQ_LENGTH = 168   # step4:53
LABEL_FEATURE = 11  # column 13 "Wind Speed 10 m Avg." minus the two id columns
HORIZONS = 3       # y1, y2, y3 (step4:14-16)


def _cuda_f32(name, t):
    if not t.is_cuda:
        raise RuntimeError(f"windgnn_b200: {name} is on {t.device}; CUDA-only (no CPU fallback)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"windgnn_b200: {name} must be float32")
    return t.contiguous()


def num_windows(n_rows: int, seq_length: int = SEQ_LENGTH, horizons: int = HORIZONS) -> int:
    return int(_lib.load().wg_num_windows(n_rows, seq_length, horizons))


def pivot_long_table(station_names, values: torch.Tensor):
    """Long table -> ``[time, station, feature]`` like step4:36-47.

    ``station_names``: one name per row of the long table (column 0 of the reference's array), any
    sequence NumPy can ``np.unique``; ``values [n_rows, F]`` the numeric columns (2:15) on the GPU, file
    order.  Stations end up in ``np.unique`` (alphabetical) order, each station's rows keep their file
    order.  Returns ``(table [Ttot, S, F], station_order)``.  The name -> rank map is host plumbing
    (strings); the data movement is the library's ``wg_pivot_table_f32``."""
    import numpy as np

    lib = _lib.load()
    values = _cuda_f32("values", values)
    if values.dim() != 2:
        raise RuntimeError("values must be [n_rows, F]")
    n_rows, F = values.shape
    stations, inverse = np.unique(np.asarray(station_names), return_inverse=True)   # step4:38
    if inverse.shape[0] != n_rows:
        raise RuntimeError(f"{inverse.shape[0]} station names for {n_rows} rows")
    S = len(stations)
    if S == 0 or n_rows % S:
        raise RuntimeError(f"{n_rows} rows do not split evenly over {S} stations (the reference's np.concatenate "
                           "along the station axis needs equal counts, step4:47)")
    Ttot = n_rows // S
    dev = values.device
    sid = torch.from_numpy(inverse.astype(np.int32)).to(dev)
    table = torch.empty((Ttot, S, F), dtype=torch.float32, device=dev)
    counts = torch.empty(S, dtype=torch.int32, device=dev)
    _lib.check(lib.wg_pivot_table_f32(sid.data_ptr(), values.data_ptr(), table.data_ptr(), counts.data_ptr(), n_rows, S,
                                      F, Ttot, dev.index or 0, torch.cuda.current_stream(dev).cuda_stream))
    c = counts.cpu()
    if int(c.min()) != Ttot or int(c.max()) != Ttot:
        raise RuntimeError(f"stations have unequal row counts ({int(c.min())} .. {int(c.max())}); the reference's "
                           "pivot (step4:47) requires them equal")
    return table, list(stations)


def create_sequences(table: torch.Tensor, seq_length: int = SEQ_LENGTH, perm: torch.Tensor | None = None,
                     label_feature: int = LABEL_FEATURE, horizons: int = HORIZONS, want_x: bool = True):
    """``table [Ttot, S, F]`` -> ``(x [N, L, S, F], y [N, L, horizons*S])`` like step4:7-22.

    ``perm`` (int64 ``[N]``) plays the role of the reference's shuffle (step4:23-26); without it
    the windows keep their chronological order and ``x`` is simply a view of the table.
    """
    lib = _lib.load()
    table = _cuda_f32("table", table)
    if table.dim() != 3:
        raise RuntimeError("table must be [time, station, feature]")
    Ttot, S, F = table.shape
    dev = table.device
    if perm is None:
        N = int(lib.wg_num_windows(Ttot, seq_length, horizons))
    else:
        if perm.dtype != torch.int64 or not perm.is_cuda:
            raise RuntimeError("perm must be a CUDA int64 tensor")
        perm = perm.contiguous()
        N = perm.numel()
        # every entry must name a complete window (the kernels index table[perm[n] * L ...] directly)
        n_valid = int(lib.wg_num_windows(Ttot, seq_length, horizons))
        if N and (int(perm.min()) < 0 or int(perm.max()) >= n_valid):
            raise RuntimeError(
                f"perm entries must lie in [0, {n_valid}) — the table holds {n_valid} complete windows of "
                f"{seq_length} rows with {horizons} label rows after them; got [{int(perm.min())}, {int(perm.max())}]")
    y = torch.empty((N, seq_length, horizons * S), dtype=torch.float32, device=dev)
    if perm is None and want_x:
        x = table[: N * seq_length].view(N, seq_length, S, F)  # zero-copy: windows are contiguous
        x_ptr = None
    else:
        x = torch.empty((N, seq_length, S, F), dtype=torch.float32, device=dev) if want_x else None
        x_ptr = x.data_ptr() if want_x else None
    if N:
        _lib.check(lib.wg_make_windows_f32(
            table.data_ptr(), perm.data_ptr() if perm is not None else None, x_ptr, y.data_ptr(),
            Ttot, S, F, seq_length, label_feature, horizons, N, dev.index or 0,
            torch.cuda.current_stream(dev).cuda_stream))
    return x, y


def window_starts(n_rows: int, seq_length: int = SEQ_LENGTH, stride: int = 1, horizons: int = 0) -> torch.Tensor:
    """CPU int64 first rows ``0, stride, 2 stride, ...`` of every window of ``seq_length`` rows that has
    ``horizons`` label rows after it in a table of ``n_rows`` rows (``GCN_GRU.forecast``).  ``stride=1``: one
    forecast per hour; ``stride=seq_length, horizons=3``: the reference's non-overlapping windows (step4:10-16),
    ``num_windows`` of them."""
    if seq_length < 1 or stride < 1 or horizons < 0:
        raise ValueError("seq_length and stride must be >= 1, horizons >= 0")
    return torch.arange(0, max(n_rows - seq_length - horizons + 1, 0), stride, dtype=torch.int64)


def forecast_targets(table: torch.Tensor, starts: torch.Tensor, seq_length: int = SEQ_LENGTH,
                     label_feature: int = LABEL_FEATURE, horizons: int = HORIZONS) -> torch.Tensor:
    """``[N, horizons * S]`` targets of each window's last step, ``y[n, k*S + s] = table[starts[n] + L + k, s,
    label_feature]``: what ``create_sequences(...)[1][:, -1]`` holds for ``starts = perm * L`` (step4:14-18), for
    any starts.  Index plumbing only, on ``table``'s device."""
    if table.dim() != 3:
        raise RuntimeError("table must be [time, station, feature]")
    if starts.dtype != torch.int64 or starts.dim() != 1:
        raise RuntimeError("starts must be a 1-D int64 tensor")
    Ttot, S, _ = table.shape
    starts = starts.to(table.device)
    if starts.numel() and (int(starts.min()) < 0 or int(starts.max()) + seq_length + horizons > Ttot):
        raise RuntimeError(f"starts must lie in [0, {Ttot - seq_length - horizons}] so that every window has "
                           f"{horizons} label rows after it")
    rows = starts[:, None] + seq_length + torch.arange(horizons, device=table.device)
    return table[rows, :, label_feature].reshape(starts.numel(), horizons * S)


def denormalise_last_step(outputs: torch.Tensor, wind_min: float, wind_max: float) -> torch.Tensor:
    """``outputs [B, T, H]`` (or ``[T, H]``) -> ``[B, H]``: ``out[:, -1] * (max - min) + min`` in
    fp32 with NumPy's rounding (main.py:103) — only ``3S`` floats per window leave the GPU."""
    lib = _lib.load()
    outputs = _cuda_f32("outputs", outputs)
    if outputs.dim() == 2:
        outputs = outputs.unsqueeze(0)
    B, T, H = outputs.shape
    pred = torch.empty((B, H), dtype=torch.float32, device=outputs.device)
    if B:
        _lib.check(lib.wg_denorm_last_step_f32(outputs.data_ptr(), pred.data_ptr(), B, T, H, float(wind_min),
                                               float(wind_max), outputs.device.index or 0,
                                               torch.cuda.current_stream(outputs.device).cuda_stream))
    return pred
