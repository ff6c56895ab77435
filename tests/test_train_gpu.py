"""GPU parity of the training step (BASELINE.json configs[4]): the library's forward-with-saved-gates,
BPTT / GEMM / GCN backward, MSE loss and Adam step — through the C-ABI — against the hand-written
NumPy oracle and against the reference module's own autograd gradients (``tests/golden/train_*.npz``).

Tolerance: ``max|g - ref| / max|ref| <= 1e-5`` per parameter tensor (the reference's own
fp32-vs-fp64 gradient noise is up to 2e-6, see the fixtures' ``grad32__*``)."""

import numpy as np
import pytest
import torch

import windgnn_b200
from conftest import golden, load_checkpoint
from oracle import normalised_max_error
from oracle.gcn_gru_oracle import PARAM_KEYS
from oracle.train_oracle import adam_step, flatten_grads, gcn_gru_loss_and_grads
from windgnn_b200 import _lib, train

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = "cuda:0"


def _model(S, sd=None, dims=None):
    m = windgnn_b200.GCN_GRU(*(dims or (13, 13, 13, 13 * S, 3 * S)))
    m.load_state_dict(sd if sd is not None else load_checkpoint(S), strict=True)
    return m.to(DEV)


def _adj(S):
    return torch.from_numpy(golden(f"adj_ref_{S}.npy").astype(np.float32)).to(DEV)


def _params(m):
    return [m.conv1.weight, m.conv1.bias, m.conv2.weight, m.conv2.bias,
            m.gru.weight_ih_l0, m.gru.weight_hh_l0, m.gru.bias_ih_l0, m.gru.bias_hh_l0]


@pytest.mark.parametrize("S", [7, 34])
def test_gradients_match_reference_autograd(S):
    """The reference's loop body (main.py:66-76) run with the drop-in module: same loss, same grads."""
    g = golden(f"train_{S}.npz")
    model = _model(S).train()
    x, y = torch.from_numpy(g["x"]).to(DEV), torch.from_numpy(g["y"]).to(DEV)
    out = model(_adj(S), x)                      # grad enabled -> GcnGruFunction
    loss = torch.nn.MSELoss()(out, y)            # main.py:49,72
    model.zero_grad()
    loss.backward()                              # main.py:76
    assert abs(loss.item() - float(g["loss"])) <= 1e-6 * abs(float(g["loss"])) + 1e-7
    for k, p in model.named_parameters():
        ref = g["grad__" + k.replace(".", "__")]
        assert p.grad is not None and p.grad.shape == ref.shape
        assert normalised_max_error(p.grad.cpu().numpy(), ref) <= TOL, k


@pytest.mark.parametrize("S", [7, 34])
def test_flat_backward_matches_oracle_with_arbitrary_upstream_gradient(S):
    g = golden(f"train_{S}.npz")
    sd = load_checkpoint(S)
    model = _model(S, sd)
    adj = _adj(S)
    x = torch.from_numpy(g["x"]).to(DEV)
    rng = np.random.default_rng(3)
    d_out = rng.standard_normal(g["y"].shape).astype(np.float32) * 1e-3
    with torch.no_grad():
        ps = [p.data for p in _params(model)]
        out, ws = train.forward_train(adj, x, ps)
        y_inf = model(adj, x)
        flat = train.backward(adj, x, ps, out, torch.from_numpy(d_out).to(DEV), ws)
        flat2 = train.backward(adj, x, ps, out, torch.from_numpy(d_out).to(DEV), ws)
    assert torch.equal(out, y_inf)               # the training forward IS the inference forward
    assert torch.equal(flat, flat2)              # fixed-order reductions: bit-reproducible
    _, _, G = gcn_gru_loss_and_grads(adj.cpu().numpy(), g["x"], g["y"], sd, dtype=np.float64, d_out=d_out)
    views = train.split_flat(flat, [tuple(sd[k].shape) for k in PARAM_KEYS])
    for k, v in zip(PARAM_KEYS, views):
        assert normalised_max_error(v.cpu().numpy(), G[k]) <= TOL, k
    assert flat.numel() == flatten_grads(G).size == _lib.load().wg_gcn_gru_param_count(S, 13, 13, 13, 3 * S)


def test_gradients_ragged_batches_and_short_windows():
    """Batch sizes that do not fill a CTA (4 / 16 / 32 sequences), T = 1 and odd T; 601 windows is past the
    switch from 4 to 16 sequences per CTA in the BPTT kernel."""
    sd = load_checkpoint(7)
    model = _model(7, sd)
    adj = _adj(7)
    rng = np.random.default_rng(11)
    for B, T in ((1, 1), (5, 3), (17, 6), (37, 9), (601, 4)):
        x = rng.random((B, T, 7, 13), dtype=np.float32)
        y = rng.random((B, T, 21), dtype=np.float32)
        with torch.no_grad():
            ps = [p.data for p in _params(model)]
            out, ws = train.forward_train(adj, torch.from_numpy(x).to(DEV), ps)
            loss, d_out = train.mse_loss_grad(out, torch.from_numpy(y).to(DEV))
            flat = train.backward(adj, torch.from_numpy(x).to(DEV), ps, out, d_out, ws)
        ref_loss, ref_out, G = gcn_gru_loss_and_grads(adj.cpu().numpy(), x, y, sd, dtype=np.float64)
        assert normalised_max_error(out.cpu().numpy(), ref_out) <= TOL
        assert abs(loss.item() - ref_loss) <= 2e-6 * ref_loss
        assert normalised_max_error(flat.cpu().numpy(), flatten_grads(G)) <= TOL, (B, T)


def test_gradients_non_default_widths():
    """F_in != F_hid != 13, H != 3S (the reference ctor allows them): the padded-16 GCN backward."""
    g = golden("fwd_rand.npz")
    sd = {k: torch.from_numpy(g[k.replace(".", "__")]) for k in PARAM_KEYS}
    S, Fin, Fh, H = 5, 6, 10, 11
    model = _model(S, sd, dims=(Fin, Fh, 13, 13 * S, H))
    adj = torch.from_numpy(g["adj"]).to(DEV)
    rng = np.random.default_rng(5)
    y = rng.random(g["y_ref_f32"].shape, dtype=np.float32)
    x = torch.from_numpy(g["x"]).to(DEV)
    out = model(adj, x)
    loss = torch.nn.MSELoss()(out, torch.from_numpy(y).to(DEV))
    loss.backward()
    ref_loss, _, G = gcn_gru_loss_and_grads(g["adj"], g["x"], y, sd, dtype=np.float64)
    assert abs(loss.item() - ref_loss) <= 2e-6 * ref_loss
    for k, p in model.named_parameters():
        assert normalised_max_error(p.grad.cpu().numpy(), G[k]) <= TOL, k


@pytest.mark.parametrize("S", [7, 34])
def test_three_adam_steps_follow_the_reference_trajectory(S):
    """Trainer.step x3 from the shipped checkpoint == the reference loop with torch.optim.Adam(lr=1e-3)."""
    g = golden(f"train_{S}.npz")
    model = _model(S).train()
    tr = train.Trainer(model, _adj(S), lr=1e-3)
    x, y = torch.from_numpy(g["x"]).to(DEV), torch.from_numpy(g["y"]).to(DEV)
    losses = [tr.step(x, y).item() for _ in range(3)]
    np.testing.assert_allclose(losses, g["losses3"], rtol=2e-5)
    sd_after = model.state_dict()
    for k in PARAM_KEYS:
        ref = g["param3__" + k.replace(".", "__")]
        start = load_checkpoint(S)[k].numpy()
        moved = np.abs(ref - start).max()
        assert moved > 0
        # compare the UPDATE (3 steps of ~lr each), not the parameter: tolerance relative to the movement.
        # Adam's step is m / sqrt(v) — sign-like — so entries whose gradient is at the fp32 noise level
        # move by a noise-dominated amount; they bound the max, the mean shows the typical agreement.
        diff = np.abs(sd_after[k].cpu().numpy() - ref)
        assert diff.max() <= 2e-2 * moved, (k, diff.max(), moved)
        assert diff.mean() <= 2e-4 * moved, (k, diff.mean(), moved)
    # state_dict keys and shapes are unchanged by the flat re-pointing
    assert list(sd_after.keys()) == list(PARAM_KEYS)


def test_adam_kernel_matches_oracle():
    lib = _lib.load()
    rng = np.random.default_rng(0)
    n = 100_003
    p = rng.standard_normal(n).astype(np.float32)
    m = np.zeros(n, np.float32)
    v = np.zeros(n, np.float32)
    tp, tm, tv = (torch.from_numpy(a.copy()).to(DEV) for a in (p, m, v))
    p64, m64, v64 = p.astype(np.float64), m.astype(np.float64), v.astype(np.float64)
    st = torch.cuda.current_stream().cuda_stream
    for step in range(1, 6):
        gr = (rng.standard_normal(n) * 10.0 ** rng.integers(-6, 1, n)).astype(np.float32)
        tg = torch.from_numpy(gr).to(DEV)
        _lib.check(lib.wg_adam_step_f32(tp.data_ptr(), tg.data_ptr(), tm.data_ptr(), tv.data_ptr(), n,
                                        1e-3, 0.9, 0.999, 1e-8, step, 0.5, 0, st))
        p64, m64, v64 = adam_step(p64, 0.5 * gr.astype(np.float64), m64, v64, step)
    torch.cuda.synchronize()
    assert normalised_max_error(tp.cpu().numpy(), p64) <= 1e-6   # fp32 parameter rounding, 5 steps
    assert normalised_max_error(tm.cpu().numpy(), m64) <= 1e-6
    assert normalised_max_error(tv.cpu().numpy(), v64) <= 1e-6


def test_full_size_training_step_properties():
    """BASELINE configs[4] per-GPU shard (512 windows of the 34-station model): the gradient of a
    batch is the mean of the gradients of its halves (linearity of the mean loss), bit-reproducible."""
    S, B = 34, 512
    model = _model(S)
    adj = _adj(S)
    gen = torch.Generator(device=DEV).manual_seed(7)
    x = torch.rand((B, 168, S, 13), generator=gen, device=DEV)
    y = torch.rand((B, 168, 3 * S), generator=gen, device=DEV)

    def grads(xs, ys):
        with torch.no_grad():
            ps = [p.data for p in _params(model)]
            out, ws = train.forward_train(adj, xs, ps)
            loss, d_out = train.mse_loss_grad(out, ys)
            return loss.item(), train.backward(adj, xs, ps, out, d_out, ws)

    l_all, g_all = grads(x, y)
    l_a, g_a = grads(x[:256], y[:256])
    l_b, g_b = grads(x[256:], y[256:])
    assert abs(l_all - 0.5 * (l_a + l_b)) <= 1e-6 * l_all
    assert normalised_max_error(g_all.cpu().numpy(), (0.5 * (g_a + g_b)).cpu().numpy()) <= TOL
    _, g_again = grads(x, y)
    assert torch.equal(g_all, g_again)
    assert torch.isfinite(g_all).all()


def test_training_rejects_what_it_does_not_support():
    model = _model(7)
    with pytest.raises(RuntimeError):
        train.forward_train(_adj(7).cpu(), torch.zeros(1, 2, 7, 13), [p.data.cpu() for p in _params(model)])
    with pytest.raises(_lib.WindGNNError) as ei:   # T = 0 is an invalid argument, not an unsupported shape
        train.forward_train(_adj(7), torch.zeros(1, 0, 7, 13, device=DEV), [p.data for p in _params(model)])
    assert ei.value.code == _lib.WG_ERR_BAD_ARG and "non-positive" in str(ei.value)
    lib = _lib.load()
    assert lib.wg_gcn_gru_train_workspace_bytes(4, 8, 7, 13, 32, 13, 21) == 0      # hidden GCN width > 16
    assert "feature widths" in _lib.last_error()
    assert lib.wg_gcn_gru_train_workspace_bytes(4, 8, 300, 13, 13, 13, 900) == 0   # H too large for the BPTT kernel
    assert lib.wg_gcn_gru_train_workspace_bytes(4, 8, 40, 13, 13, 13, 120) == 0    # W_hh no longer fits shared memory
    assert "recurrence" in _lib.last_error()


@pytest.mark.parametrize("S,H,B,T", [(1, 3, 5, 4), (3, 9, 33, 7), (12, 36, 70, 11), (20, 50, 31, 6), (35, 105, 9, 5),
                                     (9, 27, 700, 3),
                                     # gru_bwd_regw_kernel (padded hidden size 24 / 104): batches that select its
                                     # 8-, 16- and 28-sequence CTAs (the goldens above run the 4-sequence one)
                                     (7, 21, 700, 3), (7, 22, 1500, 3), (8, 24, 2500, 2),
                                     (34, 102, 700, 2), (34, 101, 1300, 2), (34, 103, 2400, 2),
                                     # gcn_bwd_kernel<13> (13-wide features, 48 < S): 60 stations, and 90 stations,
                                     # whose shared memory cuts the row block down to 2 rows
                                     (60, 30, 40, 3), (90, 45, 20, 2)])
def test_gradients_ragged_model_shapes(S, H, B, T):
    """Random models with odd station counts / hidden sizes (H odd, even-not-multiple-of-4, near the
    shared-memory limit of the recurrence), batches that end inside a CTA and inside a GEMM tile, a batch past the
    16-sequence BPTT switch, every CTA size of the register-resident BPTT kernel, and station counts past the
    row-per-lane GCN backward: every GEMM edge predicate, unaligned leading dimension and padded column is exercised."""
    torch.manual_seed(S * 100 + B)
    m = windgnn_b200.GCN_GRU(13, 13, 13, 13 * S, H)
    with torch.no_grad():
        m.conv1.weight.mul_(0.3)
        m.conv2.weight.mul_(0.3)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    rng = np.random.default_rng(B)
    adj = (rng.random((S, S), dtype=np.float32) / S).astype(np.float32)
    x = rng.random((B, T, S, 13), dtype=np.float32)
    y = rng.random((B, T, H), dtype=np.float32)
    m = m.to(DEV)
    out = m(torch.from_numpy(adj).to(DEV), torch.from_numpy(x).to(DEV))
    loss = torch.nn.MSELoss()(out.reshape(B, T, H), torch.from_numpy(y).to(DEV))
    loss.backward()
    ref_loss, _, G = gcn_gru_loss_and_grads(adj, x, y, sd, dtype=np.float64)
    assert abs(loss.item() - ref_loss) <= 2e-6 * ref_loss
    for k, p in m.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), k
        assert normalised_max_error(p.grad.cpu().numpy(), G[k]) <= TOL, k
