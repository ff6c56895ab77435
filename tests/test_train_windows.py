"""Training on windows over one table (``Trainer.step_table``, ``GCN_GRU.forward_windows``,
``wg_gcn_gru_forward_train_windows_f32`` / ``wg_gcn_gru_backward_windows_f32`` / ``wg_mse_window_labels_f32``): GCN,
input projection and their gradients once per table row, the targets read from the table.

For the non-overlapping chronological windows that ``create_sequences`` materialises every comparison with the
materialised path is exact (``torch.equal``): each table row then has one contributor, so the per-row gate gradients
are copies and every kernel sees the same rows.  Overlapping windows sum per row in another order than the
materialised path; they are held to ``max|g - ref| / max|ref| <= 1e-5`` against the float64 oracle and the
materialised path."""

import ctypes

import numpy as np
import pytest
import torch

import windgnn_b200
from conftest import golden, load_checkpoint
from oracle import normalised_max_error
from oracle.gcn_gru_oracle import PARAM_KEYS
from oracle.train_oracle import gcn_gru_loss_and_grads
from windgnn_b200 import _lib, train

TOL = 1e-5
DEV = "cuda:0"
DIMS34 = (34, 13, 13, 13, 102)   # S, F_in, F_hid, F_out, H
LABEL, K = 11, 3


# ---------------------------------------------------------------------------------------------
# host: no GPU
# ---------------------------------------------------------------------------------------------
def test_train_windows_workspace_query():
    lib = _lib.load()
    ws = lib.wg_gcn_gru_train_windows_workspace_bytes(4096, 26304, 168, *DIMS34)
    assert ws > 0
    # U (448 columns) and GI (312) of every table row, and the per-row gate gradients (408)
    assert ws >= 26304 * (448 + 312 + 408) * 4
    assert lib.wg_gcn_gru_train_windows_workspace_bytes(4096, 2097024, 168, *DIMS34) > 0
    # the training path's limits, with its texts
    for n, ttot, dims in ((512, 26304, (34, 13, 13, 13, 107)), (512, 26304, (34, 17, 13, 13, 102)),
                          (-1, 26304, DIMS34)):
        assert lib.wg_gcn_gru_train_windows_workspace_bytes(n, ttot, 168, *dims) == 0
        text = _lib.last_error()
        assert lib.wg_gcn_gru_train_workspace_bytes(n, 168, *dims) == 0
        assert _lib.last_error() == text
    assert lib.wg_gcn_gru_train_windows_workspace_bytes(4, 100, 101, *DIMS34) == 0
    assert "L <= Ttot" in _lib.last_error()
    assert lib.wg_gcn_gru_train_windows_workspace_bytes(4, 2097025, 168, *DIMS34) == 0
    assert "exceeds one pass" in _lib.last_error()
    # the entry points report the same before anything else (the pointers are never looked at)
    fake = ctypes.c_void_p(8)
    rc = lib.wg_gcn_gru_forward_train_windows_f32(*([fake] * 12), 4, 2097025, 168, *DIMS34, None, 0, 0, None)
    assert rc == _lib.WG_ERR_UNSUPPORTED and "exceeds one pass" in _lib.last_error()
    rc = lib.wg_gcn_gru_backward_windows_f32(*([fake] * 12), 512, 26304, 168, 34, 13, 13, 13, 107, None, 0, 0, None)
    assert rc == _lib.WG_ERR_UNSUPPORTED and "training: GRU hidden size 107" in _lib.last_error()


def test_bad_starts_name_the_window():
    lib = _lib.load()
    fake = ctypes.c_void_p(8)   # never dereferenced: the starts are checked first
    Ttot, L = 400, 168

    def host(a):
        return (ctypes.c_int64 * len(a))(*a)

    for entry in (lib.wg_gcn_gru_forward_train_windows_f32, lib.wg_gcn_gru_backward_windows_f32):
        rc = entry(fake, fake, None, *([fake] * 9), 2, Ttot, L, *DIMS34, fake, 1 << 30, 0, None)
        assert rc == _lib.WG_ERR_BAD_ARG and "starts is NULL" in _lib.last_error()
        rc = entry(fake, fake, host([0, -1]), *([fake] * 9), 2, Ttot, L, *DIMS34, fake, 1 << 30, 0, None)
        assert rc == _lib.WG_ERR_BAD_ARG and "starts[1] = -1" in _lib.last_error()
        rc = entry(fake, fake, host([0, 3, Ttot - L + 1]), *([fake] * 9), 3, Ttot, L, *DIMS34, fake, 1 << 30, 0, None)
        assert rc == _lib.WG_ERR_BAD_ARG and f"starts[2] = {Ttot - L + 1}" in _lib.last_error()
    # the labels need `horizons` more rows: Ttot - L is a valid window, not a valid loss
    args = (fake, fake, host([0, Ttot - L]), 2, L, Ttot, 34, 13, LABEL, K, fake, fake, fake, 1 << 20, 0, None)
    assert lib.wg_mse_window_labels_f32(*args) == _lib.WG_ERR_BAD_ARG
    assert f"starts[1] = {Ttot - L} outside [0, Ttot - L - horizons]" in _lib.last_error()
    args = (fake, fake, host([0]), 0, L, Ttot, 34, 13, LABEL, K, fake, fake, fake, 1 << 20, 0, None)
    assert lib.wg_mse_window_labels_f32(*args) == _lib.WG_ERR_BAD_ARG
    assert lib.wg_mse_window_labels_workspace_bytes(0) == 0


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
def _model(S, dims=None, sd=None):
    m = windgnn_b200.GCN_GRU(*(dims or (13, 13, 13, 13 * S, 3 * S)))
    m.load_state_dict(sd if sd is not None else load_checkpoint(S), strict=True)
    return m.to(DEV)


def _adj(S):
    return torch.from_numpy(golden(f"adj_ref_{S}.npy").astype(np.float32)).to(DEV)


def _table(Ttot, S, F=13, seed=0):
    rng = np.random.default_rng(seed)
    return rng.random((Ttot, S, F), dtype=np.float32)


def _windows(table, starts, L):
    """Materialised x [N, L, S, F] and targets y [N, L, K*S] (create_sequences' layout) of any starts."""
    s = np.asarray(starts, dtype=np.int64)
    rows = s[:, None] + np.arange(L)
    x = table[rows]
    lab = rows[:, :, None] + 1 + np.arange(K)                       # [N, L, K]
    y = table[lab, :, LABEL].reshape(len(s), L, K * table.shape[1])   # [N, L, K, S] -> k*S + s
    return x, y


def _ps(m):
    return [p.data for p in m._params()]


def _flat_views(flat, sd):
    return train.split_flat(flat, [tuple(sd[k].shape) for k in PARAM_KEYS])


@pytest.mark.gpu
@pytest.mark.parametrize("S,L,nwin", [(7, 168, 6), (34, 168, 8),      # gru_recur_regw_kernel
                                      (7, 4, 1300), (34, 2, 1300)])   # gru_recur_unit_kernel (N > 1184)
def test_chronological_windows_bit_identical_to_materialised(S, L, nwin):
    table = torch.from_numpy(_table(nwin * L + K, S, seed=S)).to(DEV)
    x, y = windgnn_b200.create_sequences(table, L)
    starts = windgnn_b200.window_starts(table.shape[0], L, stride=L, horizons=K)
    assert starts.numel() == x.shape[0] == nwin
    adj = _adj(S)
    m1, m2 = _model(S), _model(S)
    with torch.no_grad():
        out, ws = train.forward_train(adj, x, _ps(m1))
        out_t, ws_t = train.forward_train_windows(adj, table, starts, _ps(m2), L)
        assert torch.equal(out, out_t)
        loss, d_out = train.mse_loss_grad(out, y)
        loss_t, d_out_t = train.mse_window_labels(out_t, table, starts, L)
        assert torch.equal(loss, loss_t) and torch.equal(d_out, d_out_t)
        flat = train.backward(adj, x, _ps(m1), out, d_out, ws)
        flat_t = train.backward_windows(adj, table, starts, _ps(m2), out_t, d_out_t, ws_t, L)
        assert torch.equal(flat, flat_t)
    t1, t2 = train.Trainer(m1, adj), train.Trainer(m2, adj)
    for _ in range(3):
        assert torch.equal(t1.step(x, y), t2.step_table(table, starts, seq_length=L))
        assert torch.equal(t1.grads, t2.grads)
    assert torch.equal(t1.flat, t2.flat)


def _starts_variant(kind, Ttot, L):
    last = Ttot - L - K
    hourly = np.arange(last + 1)
    if kind == "hourly":
        return hourly
    if kind == "shuffled":
        return np.random.default_rng(5).permutation(hourly)
    if kind == "repeated":
        return np.array([5, 5, 5, 17, 17, 40, 0, last, last])
    return np.array([last, 0, 3, 90, 4, last - 30])   # gaps: rows no window covers


def _step_pieces(adj, table_d, starts, ps, L):
    out, ws = train.forward_train_windows(adj, table_d, starts, ps, L)
    loss, d_out = train.mse_window_labels(out, table_d, starts, L)
    return loss, train.backward_windows(adj, table_d, starts, ps, out, d_out, ws, L)


@pytest.mark.gpu
@pytest.mark.parametrize("S,kind", [(7, "hourly"), (7, "shuffled"), (7, "repeated"), (7, "gaps"), (34, "hourly"),
                                    (34, "shuffled")])
def test_overlapping_windows_match_float64(S, kind):
    L, Ttot = 24, 120
    table = _table(Ttot, S, seed=11)
    starts = _starts_variant(kind, Ttot, L)
    sd = load_checkpoint(S)
    m = _model(S, sd=sd)
    adj = _adj(S)
    table_d = torch.from_numpy(table).to(DEV)
    with torch.no_grad():
        loss, flat = _step_pieces(adj, table_d, torch.from_numpy(starts), _ps(m), L)
        x, y = _windows(table, starts, L)
        out_m, ws_m = train.forward_train(adj, torch.from_numpy(x).to(DEV), _ps(m))
        loss_m, d_m = train.mse_loss_grad(out_m, torch.from_numpy(y).to(DEV))
        flat_m = train.backward(adj, torch.from_numpy(x).to(DEV), _ps(m), out_m, d_m, ws_m)
    ref_loss, _, G = gcn_gru_loss_and_grads(adj.cpu().numpy(), x, y, sd, dtype=np.float64)
    assert abs(loss.item() - ref_loss) <= TOL * ref_loss
    assert loss.item() == loss_m.item()   # the same outputs and targets: the same loss
    for k, v, vm in zip(PARAM_KEYS, _flat_views(flat, sd), _flat_views(flat_m, sd)):
        assert normalised_max_error(v.cpu().numpy(), G[k]) <= TOL, k
        assert normalised_max_error(v.cpu().numpy(), vm.cpu().numpy().astype(np.float64)) <= TOL, k


# test_train_gpu.py::test_gradients_ragged_model_shapes' (S, H, B, T), then non-13 GCN widths
RAGGED = [(1, 3, 5, 4), (3, 9, 33, 7), (12, 36, 70, 11), (20, 50, 31, 6), (35, 105, 9, 5), (9, 27, 700, 3),
          (7, 21, 700, 3), (7, 22, 1500, 3), (8, 24, 2500, 2), (34, 102, 700, 2), (34, 101, 1300, 2),
          (34, 103, 2400, 2), (60, 30, 40, 3), (90, 45, 20, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("S,H,B,T,widths", [(*r, (13, 13, 13)) for r in RAGGED] +
                         [(10, 30, 50, 6, (5, 9, 11)), (16, 48, 40, 5, (16, 16, 16)), (6, 20, 30, 4, (3, 16, 2))])
def test_arbitrary_upstream_gradient_ragged_shapes(S, H, B, T, widths):
    Fi, Fh, Fo = widths
    torch.manual_seed(S * 100 + B)
    m = windgnn_b200.GCN_GRU(Fi, Fh, Fo, Fo * S, H)
    with torch.no_grad():
        m.conv1.weight.mul_(0.3)
        m.conv2.weight.mul_(0.3)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    rng = np.random.default_rng(B)
    adj = (rng.random((S, S), dtype=np.float32) / S).astype(np.float32)
    Ttot = T + max(B // 3, 4)                                   # the windows overlap: about 3 per table row
    table = rng.random((Ttot, S, Fi), dtype=np.float32)
    starts = rng.integers(0, Ttot - T + 1, size=B)
    d_out = rng.standard_normal((B, T, H)).astype(np.float32) * 1e-3
    adj_d, table_d = torch.from_numpy(adj).to(DEV), torch.from_numpy(table).to(DEV)
    with torch.no_grad():
        out, ws = train.forward_train_windows(adj_d, table_d, torch.from_numpy(starts), _ps(m), T)
        dd = torch.from_numpy(d_out).to(DEV)
        flat = train.backward_windows(adj_d, table_d, torch.from_numpy(starts), _ps(m), out, dd, ws, T)
        flat2 = train.backward_windows(adj_d, table_d, torch.from_numpy(starts), _ps(m), out, dd, ws, T)
    assert torch.equal(flat, flat2)   # fixed-order reductions: bit-reproducible
    x = table[starts[:, None] + np.arange(T)]
    _, out_ref, G = gcn_gru_loss_and_grads(adj, x, np.zeros((B, T, H), np.float32), sd, dtype=np.float64,
                                           d_out=d_out)
    assert normalised_max_error(out.cpu().numpy(), out_ref) <= TOL
    for k, v in zip(PARAM_KEYS, _flat_views(flat, sd)):
        assert torch.isfinite(v).all(), k
        assert normalised_max_error(v.cpu().numpy(), G[k]) <= TOL, k


@pytest.mark.gpu
def test_forward_windows_autograd_and_no_grad():
    S, L, Ttot = 7, 24, 90
    table = _table(Ttot, S, seed=2)
    table_d = torch.from_numpy(table).to(DEV)
    starts = torch.from_numpy(_starts_variant("shuffled", Ttot, L))
    adj = _adj(S)
    m = _model(S).train()
    out = m.forward_windows(adj, table_d, starts, seq_length=L)
    _, y = _windows(table, starts.numpy(), L)
    loss = torch.nn.MSELoss()(out, torch.from_numpy(y).to(DEV))
    m.zero_grad()
    loss.backward()
    with torch.no_grad():
        _, flat = _step_pieces(adj, table_d, starts, _ps(m), L)
    sd = m.state_dict()
    for (k, p), v in zip(m.named_parameters(), _flat_views(flat, sd)):
        assert normalised_max_error(p.grad.cpu().numpy(), v.cpu().numpy().astype(np.float64)) <= TOL, k
    with torch.no_grad():
        o = m.forward_windows(adj, table_d, seq_length=L, stride=7)   # default starts: every 7th window
        s = windgnn_b200.window_starts(Ttot, L, 7)
        assert o.shape == (s.numel(), L, 3 * S)
        for n in (0, 3, s.numel() - 1):
            w = table_d[int(s[n]):int(s[n]) + L].unsqueeze(0)
            assert torch.equal(o[n], m(adj, w))
    # the training path's limits, as forward's
    csr = windgnn_b200.CsrGraph(*windgnn_b200.ops.dense_to_csr(adj), S)
    with pytest.raises(RuntimeError, match="training is implemented for dense graphs"):
        m.forward_windows(csr, table_d, starts, seq_length=L)


@pytest.mark.gpu
def test_uneven_shards_weighted_like_one_process():
    S, L, Ttot = 7, 24, 100
    table_d = torch.from_numpy(_table(Ttot, S, seed=4)).to(DEV)
    starts = torch.from_numpy(_starts_variant("shuffled", Ttot, L))
    N = starts.numel()
    adj = _adj(S)
    tr = train.Trainer(_model(S), adj, lr=0.0)   # lr = 0: the parameters stay put, tr.grads holds each gradient
    tr.step_table(table_d, starts, seq_length=L)
    g_all = tr.grads.clone()
    parts = []
    for shard in (starts[:13], starts[13:]):
        assert train.shard_weight(shard.numel(), N) == shard.numel() / N
        tr.step_table(table_d, shard, seq_length=L, global_batch=N)
        parts.append(tr.grads.clone())
    g = (parts[0] + parts[1]).cpu().numpy()
    assert normalised_max_error(g, g_all.cpu().numpy().astype(np.float64)) <= TOL
