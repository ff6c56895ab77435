"""Tensor-core path (``precision = "tensor"``) at operand scales the shipped checkpoints never reach.

The path splits every fp32 operand into two fp16 parts.  Its error has to be as scale-free as the FP32 path's: a
model whose GCN output is small and whose W_ih is large (or the reverse), a model with small GRU weights, and inputs
in raw physical units all get the FP32 path's accuracy against the float64 oracle.  Power-of-two rescalings that
leave the GRU input gates unchanged in exact arithmetic must leave the output unchanged bit for bit.
"""

import functools

import numpy as np
import pytest
import torch

import windgnn_b200
from conftest import golden, load_checkpoint
from oracle import gcn_gru_forward, gcn_layer, normalised_max_error

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = "cuda:0"
FP16_MAX = 65504.0
PRECISIONS = ("fp32", "tensor")
ACT_FLOOR = 0.04   # output size below which the activations' absolute error (~1e-7) dominates: see test_small_signal_gru


def _state(name):
    """(module dims, state_dict, dense adjacency) of a test model: the shipped checkpoints, or the 300-station kNN
    model with F_hid = 128 and H = 128 that runs the CSR graph path."""
    if name in ("S7", "S34"):
        S = int(name[1:])
        return (13, 13, 13, 13 * S, 3 * S), load_checkpoint(S), golden(f"adj_ref_{S}.npy").astype(np.float32)
    torch.manual_seed(6)
    m = windgnn_b200.GCN_GRU(13, 128, 13, 13 * 300, 128)
    with torch.no_grad():
        m.conv1.weight.mul_(0.05)
        m.conv2.weight.mul_(0.05)
    ll = windgnn_b200.synthetic_coordinates(300, seed=9, device=DEV).cpu().numpy()
    adj = windgnn_b200.knn_graph_from_latlon(ll, k=8, device=DEV).cpu().numpy().astype(np.float32)
    return (13, 128, 13, 13 * 300, 128), {k: v.detach().clone() for k, v in m.state_dict().items()}, adj


def _model(dims, sd, precision, chunk=0):
    m = windgnn_b200.GCN_GRU(*dims)
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval()
    m.precision = precision
    m.chunk = chunk
    return m


def _rescaled(sd, k):
    """conv2 x 2^-k and W_ih x 2^k: U scales by 2^-k (ReLU is positively homogeneous), the input gates not at all."""
    out = {n: v.clone() for n, v in sd.items()}
    for n in ("conv2.weight", "conv2.bias"):
        out[n] = out[n] * 2.0 ** -k
    out["gru.weight_ih_l0"] = out["gru.weight_ih_l0"] * 2.0 ** k
    return out


@functools.lru_cache(maxsize=None)
def _case(name):
    dims, sd, adj = _state(name)
    S = adj.shape[0]
    rng = np.random.default_rng(S)
    x = rng.random((6, 24, S, 13), dtype=np.float32)
    table = torch.from_numpy(rng.random((60, S, 13), dtype=np.float32)).to(DEV)
    starts = windgnn_b200.window_starts(60, 12, 4)
    # the largest |U| of these inputs (float64 oracle) and the largest |W_ih|: where the rescaling leaves fp16
    u = gcn_layer(adj.astype(np.float64), gcn_layer(adj.astype(np.float64), x.astype(np.float64),
                                                    sd["conv1.weight"].double().numpy(),
                                                    sd["conv1.bias"].double().numpy()),
                  sd["conv2.weight"].double().numpy(), sd["conv2.bias"].double().numpy())
    umax, wmax = float(np.abs(u).max()), float(sd["gru.weight_ih_l0"].abs().max())
    top = 16
    while umax * 2.0 ** -top <= FP16_MAX and wmax * 2.0 ** top <= FP16_MAX:
        top += 1
    return dims, sd, adj, x, table, starts, top


@functools.lru_cache(maxsize=None)
def _outputs(name, k, precision):
    """(forward, forecast) of the model rescaled by 2^k, on the CPU."""
    dims, sd, adj, x, table, starts, top = _case(name)
    m = _model(dims, _rescaled(sd, k) if k else sd, precision)
    a = torch.from_numpy(adj).to(DEV)
    with torch.no_grad():
        y = m(a, torch.from_numpy(x).to(DEV))
        f = m.forecast(a, table, starts, seq_length=12)
    torch.cuda.synchronize()
    return y.cpu(), f.cpu()


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("k", [-12, -8, -4, 4, 8, 12, "top"])
@pytest.mark.parametrize("name", ["S7", "S34", "csr300"])
def test_power_of_two_rescaling_is_exact(name, k, precision):
    """Every operation only moves exponents, so the output is bit-identical to the unscaled model's, for the
    forward and for a forecast.  "top": the smallest k >= 16 at which a scaled operand (|U| 2^-k or |W_ih| 2^k)
    exceeds the fp16 range."""
    top = _case(name)[-1]
    if k == "top":
        k = top
        assert k >= 16
    y0, f0 = _outputs(name, 0, precision)
    y, f = _outputs(name, k, precision)
    assert torch.isfinite(y).all() and torch.isfinite(f).all()
    assert torch.equal(y, y0), f"k={k}: max|dy| = {float((y - y0).abs().max()):.3g}"
    assert torch.equal(f, f0), f"k={k}: max|df| = {float((f - f0).abs().max()):.3g}"


def test_top_rescaling_leaves_the_fp16_range():
    """The premise of the "top" cases: for the shipped 34-station model k = 16 already pushes an operand past fp16."""
    assert _case("S34")[-1] == 16


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("k", [0, 4, 8, 10])
@pytest.mark.parametrize("S", [7, 34])
def test_small_signal_gru(S, k, precision):
    """W_ih, W_hh, b_ih, b_hh x 2^-k: small states, a nearly linear GRU, so the recurrent product's operands (W_hh
    and h) carry the result.  H = 21 / 102 runs the tensor-core recurrence.

    Both paths evaluate sigmoid and tanh with ex2.approx (wg_common.cuh), whose error is absolute, about 1e-7
    whatever the size of the output.  At k = 8, 10 the outputs are 0.003 .. 0.02 and that floor alone reaches 1e-5 of
    them, so the error is normalised by max(max|ref|, ACT_FLOOR): the bar is the usual 1e-5 relative one wherever the
    output is at least ACT_FLOOR (k = 0, 4) and 4e-7 absolute below it."""
    sd = {n: v.clone() for n, v in load_checkpoint(S).items()}
    for n in ("gru.weight_ih_l0", "gru.weight_hh_l0", "gru.bias_ih_l0", "gru.bias_hh_l0"):
        sd[n] = sd[n] * 2.0 ** -k
    adj = golden(f"adj_ref_{S}.npy").astype(np.float32)
    x = golden(f"fwd_{S}.npz")["x"]
    ref = gcn_gru_forward(adj, x, sd, dtype=np.float64)
    m = _model((13, 13, 13, 13 * S, 3 * S), sd, precision)
    with torch.no_grad():
        y = m(torch.from_numpy(adj).to(DEV), torch.from_numpy(x).to(DEV)).cpu().numpy()
    assert np.isfinite(y).all()
    err = float(np.abs(y.astype(np.float64) - ref).max() / max(np.abs(ref).max(), ACT_FLOOR))
    assert err <= TOL, err


@pytest.mark.parametrize("precision", PRECISIONS)
def test_raw_unit_inputs(precision):
    """Inputs in physical units (pressure in Pa): x in [0, 1e5), so U and the input gates are far outside fp16."""
    S = 34
    sd = load_checkpoint(S)
    adj = golden(f"adj_ref_{S}.npy").astype(np.float32)
    x = (np.random.default_rng(5).random((4, 48, S, 13)) * 1e5).astype(np.float32)
    ref = gcn_gru_forward(adj, x, sd, dtype=np.float64)
    m = _model((13, 13, 13, 13 * S, 3 * S), sd, precision)
    with torch.no_grad():
        y = m(torch.from_numpy(adj).to(DEV), torch.from_numpy(x).to(DEV)).cpu().numpy()
    assert np.isfinite(y).all()
    err = normalised_max_error(y, ref)
    assert err <= TOL, err
