"""Host-side behaviour of the drop-in modules (no GPU): parameter names, checkpoint loading,
the CUDA-only contract, and shape inference of the registered custom ops."""

import pytest
import torch

import windgnn_b200
from conftest import load_checkpoint

REFERENCE_KEYS = [
    "conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias",
    "gru.weight_ih_l0", "gru.weight_hh_l0", "gru.bias_ih_l0", "gru.bias_hh_l0",
]


@pytest.mark.parametrize("S", [7, 34])
def test_shipped_checkpoints_load_unchanged(S):
    model = windgnn_b200.GCN_GRU(13, 13, 13, 13 * S, 3 * S)  # main.py:39-42
    assert list(model.state_dict().keys()) == REFERENCE_KEYS
    sd = load_checkpoint(S)
    result = model.load_state_dict(sd, strict=True)
    assert not result.missing_keys and not result.unexpected_keys
    for k in REFERENCE_KEYS:
        assert torch.equal(model.state_dict()[k], sd[k])


def test_parameters_reach_the_library_in_state_dict_order():
    model = windgnn_b200.GCN_GRU(13, 13, 13, 91, 21)
    named = dict(model.named_parameters())
    assert list(windgnn_b200.ops.PARAM_NAMES) == REFERENCE_KEYS
    assert all(p is named[n] for n, p in zip(REFERENCE_KEYS, model._params(), strict=True))


def test_graph_conv_layer_init_matches_reference_shapes():
    layer = windgnn_b200.GraphConvLayer(13, 5)
    assert layer.weight.shape == (13, 5) and layer.bias.shape == (5,)
    assert torch.count_nonzero(layer.bias) == 0  # step5:9


def test_no_cpu_fallback():
    model = windgnn_b200.GCN_GRU(13, 13, 13, 91, 21)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        model(torch.eye(7), torch.zeros(1, 4, 7, 13))
    with pytest.raises(RuntimeError, match="CUDA-only"):
        windgnn_b200.GraphConvLayer(13, 13)(torch.eye(7), torch.zeros(4, 7, 13))
    with pytest.raises(RuntimeError):
        model(torch.eye(7), torch.zeros(4, 7, 13))  # 3-D input: the reference raises too (step6:20)


def test_custom_ops_registered_with_shape_inference():
    x = torch.empty(5, 9, 7, 13, device="meta")
    adj = torch.empty(7, 7, device="meta")
    w = torch.empty(13, 13, device="meta")
    b = torch.empty(13, device="meta")
    out = torch.ops.windgnn.gcn_gru_forward(
        adj, x, w, b, w, b, torch.empty(63, 91, device="meta"), torch.empty(63, 21, device="meta"),
        torch.empty(63, device="meta"), torch.empty(63, device="meta"), 0,
    )
    assert out.shape == (5, 9, 21)
    assert torch.ops.windgnn.gcn_layer(adj, x, w, b).shape == (5, 9, 7, 13)


def test_mercator_matches_oracle_bitwise():
    import numpy as np

    from conftest import station_latlon
    from oracle.graph_oracle import mercator as oracle_mercator

    ll = station_latlon(34)
    assert np.array_equal(windgnn_b200.mercator(ll), oracle_mercator(ll))


def test_gradients_wrt_data_are_refused_up_front():
    """The reference never differentiates w.r.t. its data (main.py:66-77) and the library has no such
    gradient: asking for one fails immediately instead of silently returning None."""
    model = windgnn_b200.GCN_GRU(13, 13, 13, 91, 21)
    with pytest.raises(RuntimeError, match="attr_matrix / adj_matrix"):
        model(torch.eye(7), torch.zeros(1, 4, 7, 13, requires_grad=True))


@pytest.mark.gpu
def test_untrainable_paths_run_forward_and_explain_at_backward():
    """The reference module trains at any size; here training exists for dense graphs with <= 128 stations and
    GCN widths <= 16.  Elsewhere the forward still works under grad mode (as main.py:66 calls it) and
    backward() fails with the reason instead of 'autograd not implemented'."""
    dev = "cuda:0"
    layer = windgnn_b200.GraphConvLayer(13, 13).to(dev)
    out = layer(torch.eye(7, device=dev), torch.rand(4, 7, 13, device=dev))
    assert out.requires_grad and out.shape == (4, 7, 13)
    with pytest.raises(RuntimeError, match="no autograd formula"):
        out.sum().backward()
    wide = windgnn_b200.GCN_GRU(13, 32, 13, 13 * 7, 21).to(dev)   # hidden width 32: the CSR path
    y = wide(torch.eye(7, device=dev), torch.rand(2, 4, 7, 13, device=dev))
    assert y.shape == (2, 4, 21)
    with pytest.raises(RuntimeError, match="training is implemented for dense graphs"):
        y.sum().backward()
    with torch.no_grad():
        y2 = wide(torch.eye(7, device=dev), torch.rand(2, 4, 7, 13, device=dev))
    assert not y2.requires_grad
