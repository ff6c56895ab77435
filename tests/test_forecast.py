"""Rolling forecasts (``GCN_GRU.forecast``, ``wg_gcn_gru_forecast[_csr]_f32``): the last hidden state of windows over
one table, GCN and input projection once per table row.  Every GPU comparison against the forward on the
materialised windows is exact (``torch.equal``): the per-row values are the same arithmetic, and the recurrence runs
the kernel the forward would choose."""

import ctypes

import numpy as np
import pytest
import torch

import windgnn_b200
from conftest import golden, load_checkpoint
from windgnn_b200 import _lib, ops

DEV = "cuda:0"
TC = _lib.FLAG_TENSOR_CORES
DIMS34 = (34, 13, 13, 13, 102)   # S, F_in, F_hid, F_out, H


# ---------------------------------------------------------------------------------------------
# host: no GPU
# ---------------------------------------------------------------------------------------------
def test_window_starts():
    assert windgnn_b200.window_starts(10, 3).tolist() == list(range(8))
    assert windgnn_b200.window_starts(10, 3, stride=2, horizons=1).tolist() == [0, 2, 4, 6]
    for n_rows in (168, 170, 171, 2000, 26304):
        s = windgnn_b200.window_starts(n_rows, 168, stride=168, horizons=3)
        assert s.dtype == torch.int64 and s.device.type == "cpu"
        assert s.numel() == windgnn_b200.num_windows(n_rows, 168, 3)
        assert s.tolist() == [168 * n for n in range(s.numel())]
    assert windgnn_b200.window_starts(26304, 168).numel() == 26304 - 167
    assert windgnn_b200.window_starts(100, 168).numel() == 0
    assert windgnn_b200.window_starts(169, 168, horizons=3).numel() == 0
    with pytest.raises(ValueError):
        windgnn_b200.window_starts(100, 10, stride=0)


def test_forecast_workspace_query():
    lib = _lib.load()
    for flags in (0, TC):
        ws = lib.wg_gcn_gru_forecast_workspace_bytes(26134, 26304, 168, *DIMS34, 0, flags)
        assert ws > 0
        # the input-gate values of every table row are held at once (3H = 306 columns, padded to 312)
        assert ws >= 26304 * 312 * 4
    assert lib.wg_gcn_gru_forecast_csr_workspace_bytes(69, 80, 12, 300, 13, 128, 13, 128, 0, TC) > 0
    for args, text in (((10, 100, 101), "L <= Ttot"), ((10, 100, 0), "1 <= L"), ((-1, 100, 10), "N >= 0")):
        assert lib.wg_gcn_gru_forecast_workspace_bytes(*args, *DIMS34, 0, 0) == 0
        assert text in _lib.last_error()
        assert lib.wg_gcn_gru_forecast_csr_workspace_bytes(*args, *DIMS34, 0, 0) == 0
    assert lib.wg_gcn_gru_forecast_workspace_bytes(10, 200, 168, *DIMS34, 0, 8) == 0
    assert "unknown flags" in _lib.last_error()


# the shapes of test_abi.py::test_kernel_limits_are_checked_at_planning, as (N, L, S, F_in, F_hid, F_out, H, chunk,
# flags): the forecast plans them as the forward does (T = L, B = N) and gives the forward's reason
@pytest.mark.parametrize("csr,dims,reason", [
    (False, (4, 168, 7, 20, 20, 13, 21, 0, 0), "GCN feature width 20 > 16"),
    (False, (4, 8, 520, 16, 16, 16, 21, 0, 0), "S=520 too large for the dense GCN kernel"),
    (False, (4, 8, 600, 13, 13, 13, 21, 0, 0), "S=600 too large for the dense GCN kernel"),
    (False, (4, 8, 200, 16, 16, 16, 21, 0, 0), "dense GCN needs"),
    (False, (4, 8, 34, 13, 13, 13, 400, 0, 0), "GRU hidden size 400: state does not fit"),
    (True, (2, 3, 4, 20, 20, 13, 12, 0, 0), "sparse GCN: F_in / F_out must be <= 16 (got 20 / 13)"),
    (True, (2, 3, 300, 13, 2000, 13, 24, 0, 0), "sparse GCN: hidden width 2000 too large"),
    (True, (20000, 168, 300, 13, 32, 13, 24, 20000, 0), "sparse GCN: chunk of 3360000 rows too large"),
    (True, (2, 3, 300, 13, 32, 13, 400, 0, 0), "GRU hidden size 400: state does not fit"),
])
def test_forecast_rejects_what_the_forward_rejects(csr, dims, reason):
    lib = _lib.load()
    N, L = dims[:2]
    fdims = (N, L + 5, *dims[1:])   # N, Ttot, L, ...
    query, entry, n_ptrs = ((lib.wg_gcn_gru_forecast_csr_workspace_bytes, lib.wg_gcn_gru_forecast_csr_f32, 14) if csr
                            else (lib.wg_gcn_gru_forecast_workspace_bytes, lib.wg_gcn_gru_forecast_f32, 12))
    assert query(*fdims) == 0
    assert reason in _lib.last_error()
    fake = ctypes.c_void_p(8)   # never dereferenced: planning fails first
    assert entry(*([fake] * n_ptrs), *fdims, None, 0, 0, None) == _lib.WG_ERR_UNSUPPORTED
    assert reason in _lib.last_error()


def test_forecast_validates_starts_before_anything_launches():
    lib = _lib.load()
    fake = ctypes.c_void_p(8)   # device pointers: never dereferenced; the workspace stays NULL so nothing can launch
    Ttot, L = 200, 168
    dims = (Ttot, L, *DIMS34, 0, 0)
    for bad, n_bad in ((-1, 2), (Ttot - L + 1, 1)):
        starts = (ctypes.c_int64 * 3)(0, Ttot - L, 0)
        starts[n_bad] = bad
        for csr in (False, True):
            entry, n_dev = (lib.wg_gcn_gru_forecast_csr_f32, 4) if csr else (lib.wg_gcn_gru_forecast_f32, 2)
            ptrs = [fake] * n_dev + [ctypes.cast(starts, ctypes.c_void_p)] + [fake] * 9
            assert entry(*ptrs, 3, *dims, None, 0, 0, None) == _lib.WG_ERR_BAD_ARG
            assert f"starts[{n_bad}] = {bad} outside" in _lib.last_error()
    rc = lib.wg_gcn_gru_forecast_f32(fake, fake, None, *([fake] * 9), 3, *dims, None, 0, 0, None)
    assert rc == _lib.WG_ERR_BAD_ARG and "starts is NULL" in _lib.last_error()
    # valid starts, NULL workspace: rejected as such
    ok = (ctypes.c_int64 * 2)(0, Ttot - L)
    rc = lib.wg_gcn_gru_forecast_f32(fake, fake, ctypes.cast(ok, ctypes.c_void_p), *([fake] * 9), 2, *dims, None, 0,
                                     0, None)
    assert rc == _lib.WG_ERR_WORKSPACE
    # N == 0 is a valid no-op
    assert lib.wg_gcn_gru_forecast_f32(*([None] * 12), 0, *dims, None, 0, 0, None) == _lib.WG_OK
    assert lib.wg_gcn_gru_forecast_csr_f32(*([None] * 14), 0, *dims, None, 0, 0, None) == _lib.WG_OK


def test_fake_registration_gives_the_shapes():
    S, Fh, H, Ttot, N = 34, 13, 102, 500, 77
    m = lambda *shape, dtype=torch.float32: torch.empty(shape, dtype=dtype, device="meta")  # noqa: E731
    params = (m(13, Fh), m(Fh), m(Fh, 13), m(13), m(3 * H, 13 * S), m(3 * H, H), m(3 * H), m(3 * H))
    starts = m(N, dtype=torch.int64)
    out = ops.gcn_gru_forecast(m(S, S), m(Ttot, S, 13), starts, *params, 168)
    assert out.shape == (N, H) and out.device.type == "meta" and out.dtype == torch.float32
    csr = (m(S + 1, dtype=torch.int32), m(200, dtype=torch.int32), m(200))
    out = ops.gcn_gru_forecast_csr(*csr, m(Ttot, S, 13), starts, *params, 168, 0, TC)
    assert out.shape == (N, H) and out.device.type == "meta"


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
def _params(m):
    return [p.detach() for p in (m.conv1.weight, m.conv1.bias, m.conv2.weight, m.conv2.bias, m.gru.weight_ih_l0,
                                 m.gru.weight_hh_l0, m.gru.bias_ih_l0, m.gru.bias_hh_l0)]


def _shipped(S):
    m = windgnn_b200.GCN_GRU(13, 13, 13, 13 * S, 3 * S)
    m.load_state_dict(load_checkpoint(S), strict=True)
    adj = torch.from_numpy(golden(f"adj_ref_{S}.npy").astype(np.float32)).to(DEV)
    return m.to(DEV).eval(), adj


def _random(S, H, Fh=13, seed=0, scale=0.3):
    torch.manual_seed(seed)
    m = windgnn_b200.GCN_GRU(13, Fh, 13, 13 * S, H)
    with torch.no_grad():
        m.conv1.weight.mul_(scale)
        m.conv2.weight.mul_(scale)
    rng = np.random.default_rng(seed)
    adj = torch.from_numpy((rng.random((S, S), dtype=np.float32) / S).astype(np.float32)).to(DEV)
    return m.to(DEV).eval(), adj


def _table(Ttot, S, seed=1):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.rand((Ttot, S, 13), generator=g, device=DEV)


def _materialise(table, starts, L):
    idx = starts.to(table.device)[:, None] + torch.arange(L, device=table.device)
    return table[idx]   # [N, L, S, F]


def _check(m, adj, table, starts, L, flags, chunk=0):
    """forecast == the forward's last step on the materialised windows (same chunk and flags), bit for bit."""
    m.chunk = chunk
    m.precision = "tensor" if flags else "fp32"
    got = m.forecast(adj, table, starts, seq_length=L)
    x = _materialise(table, starts, L)
    csr = m._csr_of(adj)
    with torch.no_grad():
        if csr is None:
            want = ops.gcn_gru_forward(adj, x, *_params(m), chunk, flags)[:, -1]
        else:
            want = ops.gcn_gru_forward_csr(*csr, x, *_params(m), chunk, flags)[:, -1]
    torch.cuda.synchronize()
    assert got.shape == want.shape == (starts.numel(), m.gru.weight_hh_l0.shape[1])
    assert torch.isfinite(got).all()
    assert torch.equal(got, want)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, TC])
@pytest.mark.parametrize("S", [7, 34])
def test_all_hourly_windows_of_the_shipped_models(S, flags):
    """Every stride-1 window of a 2,000-row table: 1,833 windows > 1,184, the throughput recurrence kernels."""
    m, adj = _shipped(S)
    table = _table(2000, S)
    starts = windgnn_b200.window_starts(2000, 168)
    assert starts.numel() == 1833
    _check(m, adj, table, starts, 168, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, TC])
@pytest.mark.parametrize("S", [7, 34])
def test_small_batches_run_the_register_resident_recurrence(S, flags):
    """N <= 1,184 windows of H = 21 / 102: gru_recur_regw_kernel on the FP32 path (CTAs of 1 .. 4 windows)."""
    m, adj = _shipped(S)
    table = _table(700, S, seed=2)
    for N in (1, 3, 300, 1184):
        starts = torch.randint(0, 700 - 168 + 1, (N,), generator=torch.Generator().manual_seed(N))
        _check(m, adj, table, starts, 168, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, TC])
def test_generic_hidden_size_unit_kernel(flags):
    """H = 50: the generic (runtime-H) gru_recur_unit_kernel, N > 1,184."""
    m, adj = _random(10, 50, seed=4)
    table = _table(1400, 10, seed=3)
    _check(m, adj, table, windgnn_b200.window_starts(1400, 24), 24, flags)


@pytest.mark.gpu
def test_wide_hidden_size_column_tiled_kernel():
    """S = 50, H = 150: gru_recur_kernel (W_hh^T through L1 / L2; the forward stages its stores, the forecast does
    not store them)."""
    m, adj = _random(50, 150, seed=5)
    table = _table(160, 50, seed=4)
    _check(m, adj, table, windgnn_b200.window_starts(160, 20), 20, 0)
    _check(m, adj, table, torch.tensor([140, 3, 77, 3]), 20, 0)


def _knn300():
    ll = windgnn_b200.synthetic_coordinates(300, seed=9, device=DEV).cpu().numpy()
    return windgnn_b200.knn_graph_csr_from_latlon(ll, k=8, device=DEV), windgnn_b200.knn_graph_from_latlon(
        ll, k=8, device=DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("Fh,H,flags", [(128, 128, 0), (128, 128, TC), (320, 48, 0), (320, 48, TC)])
def test_csr_graph(Fh, H, flags):
    """300 stations (kNN): the CSR path — gcn_sparse_plan_kernel at hidden width 128, the lane kernels above 256;
    the CsrGraph object and the dense matrix (converted through the cache) give the same result."""
    csr, dense = _knn300()
    m, _ = _random(300, H, Fh=Fh, seed=6, scale=0.05)
    table = _table(80, 300, seed=5)
    starts = windgnn_b200.window_starts(80, 12)
    got = _check(m, csr, table, starts, 12, flags)
    assert torch.equal(got, _check(m, dense, table, starts, 12, flags))


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, TC])
def test_ragged_starts_and_lengths(flags):
    m, adj = _shipped(34)
    Ttot = 700
    table = _table(Ttot, 34, seed=6)
    gen = torch.Generator().manual_seed(7)
    rand = torch.randint(0, Ttot - 168 + 1, (50,), generator=gen)
    rand[10:13] = rand[3]                                                       # duplicates
    _check(m, adj, table, rand, 168, flags)                                     # unsorted, random, duplicates
    _check(m, adj, table, torch.tensor([Ttot - 168, 0]), 168, flags)            # both ends of the table
    _check(m, adj, table, windgnn_b200.window_starts(Ttot, 1), 1, flags)        # L = 1
    _check(m, adj, table, windgnn_b200.window_starts(Ttot, 37, stride=3), 37, flags)   # odd L
    _check(m, adj, table, torch.randint(100, 201, (40,), generator=gen), 168, flags)    # span inside the table
    # small chunk: GCN + projection in pieces of 7 x 168 rows, the recurrence in 8 passes
    _check(m, adj, table, rand, 168, flags, chunk=7)
    _check(m, adj, table, torch.randint(0, Ttot - 19, (1300,), generator=gen), 19, flags, chunk=600)


@pytest.mark.gpu
def test_anchored_to_the_reference_windows():
    """starts = perm * L: the reference's shuffled non-overlapping windows (step4:10-26) and its evaluation
    (main.py:101-116)."""
    from oracle import gcn_gru_forward, normalised_max_error

    m, adj = _shipped(34)
    L, Ttot = 168, 2000
    table = _table(Ttot, 34, seed=8)
    n = windgnn_b200.num_windows(Ttot, L, 3)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(3)).to(DEV)
    x, y = windgnn_b200.create_sequences(table, L, perm)
    r = (0.25, 17.5)
    for precision in ("fp32", "tensor"):
        m.precision = precision
        got = m.forecast(adj, table, perm * L, seq_length=L, last_step_range=r)
        with torch.no_grad():
            want = windgnn_b200.denormalise_last_step(m(adj, x), *r)
        assert torch.equal(got, want)
    m.precision = "fp32"
    h = m.forecast(adj, table, (perm * L)[:3], seq_length=L).cpu().numpy()
    ref = gcn_gru_forward(adj.cpu().numpy(), x[:3].cpu().numpy(), load_checkpoint(34), dtype=np.float32)[:, -1]
    assert normalised_max_error(h, ref) <= 1e-5
    assert torch.equal(windgnn_b200.forecast_targets(table, perm * L, L), y[:, -1])
    assert torch.equal(windgnn_b200.forecast_targets(table, (perm * L).cpu(), L), y[:, -1])


@pytest.mark.gpu
def test_streams_and_grad_mode():
    m, adj = _shipped(7)
    table = _table(1500, 7, seed=9)
    starts = windgnn_b200.window_starts(1500, 168)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        a = m.forecast(adj, table, starts)
    with torch.cuda.stream(s2):
        b = m.forecast(adj, table, starts.to(DEV))   # starts on the GPU are read back to the host
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    assert any(p.requires_grad for p in m.parameters())
    with torch.enable_grad():
        c = m.forecast(adj, table, starts)
    assert not c.requires_grad and torch.equal(c, a)
