"""Argument checks of the Python entry points over the C-ABI: the four GCN_GRU custom ops,
``ops.gcn_gru_forward_host``, ``train.forward_train`` and ``train.backward``.  Each must reject a bad
tensor with a message that names it before anything reaches the library, and keep its empty-input
behaviour."""

import pytest
import torch

import windgnn_b200
from windgnn_b200 import _lib, ops, train

S, F, FH, H, L = 4, 13, 13, 6, 3
PARAMS = (   # state_dict order
    ("conv1.weight", (F, FH)), ("conv1.bias", (FH,)), ("conv2.weight", (FH, F)), ("conv2.bias", (F,)),
    ("gru.weight_ih_l0", (3 * H, S * F)), ("gru.weight_hh_l0", (3 * H, H)), ("gru.bias_ih_l0", (3 * H,)),
    ("gru.bias_hh_l0", (3 * H,)),
)
NAMES = [n for n, _ in PARAMS]
DEV = "cuda:0"


def _inputs(dev, B=2, T=5, Ttot=7, n_starts=2):
    g = torch.Generator().manual_seed(0)
    d = {
        "params": [(0.1 * torch.randn(shp, generator=g)).to(dev) for _, shp in PARAMS],
        "adj": torch.full((S, S), 1.0 / S).to(dev),
        # the same all-ones / S graph in CSR form
        "csr": (torch.arange(0, S * S + 1, S, dtype=torch.int32).to(dev),
                torch.arange(S, dtype=torch.int32).repeat(S).to(dev), torch.full((S * S,), 1.0 / S).to(dev)),
        "x": torch.rand((B, T, S, F), generator=g).to(dev),
        "table": torch.rand((Ttot, S, F), generator=g).to(dev),
        "starts": torch.arange(n_starts, dtype=torch.int64),
    }
    if torch.device(dev).type == "cuda" and B > 0 and T > 0:
        d["out"], d["ws"] = train.forward_train(d["adj"], d["x"], d["params"])
    else:
        d["out"], d["ws"] = torch.zeros((B, T, H), device=dev), torch.empty(0, dtype=torch.uint8, device=dev)
    return d


ENTRY_POINTS = {
    "forward": lambda d: ops.gcn_gru_forward(d["adj"], d["x"], *d["params"]),
    "forward_csr": lambda d: ops.gcn_gru_forward_csr(*d["csr"], d["x"], *d["params"]),
    "forecast": lambda d: ops.gcn_gru_forecast(d["adj"], d["table"], d["starts"], *d["params"], L),
    "forecast_csr": lambda d: ops.gcn_gru_forecast_csr(*d["csr"], d["table"], d["starts"], *d["params"], L),
    "forward_host": lambda d: ops.gcn_gru_forward_host(d["adj"], d["x"].cpu(), d["params"]),
    "forward_train": lambda d: train.forward_train(d["adj"], d["x"], d["params"]),
    "backward": lambda d: train.backward(d["adj"], d["x"], d["params"], d["out"], d["out"], d["ws"]),
}
CSR_OPS = ("forward_csr", "forecast_csr")
FORECASTS = ("forecast", "forecast_csr")


class _Spy:
    """Stands in for the loaded library and records which of its symbols a call looked up."""

    def __init__(self, lib):
        self.lib, self.names = lib, []

    def __getattr__(self, name):
        self.names.append(name)
        return getattr(self.lib, name)


@pytest.fixture
def spy(monkeypatch):
    s = _Spy(_lib.load())
    monkeypatch.setattr(_lib, "load", lambda: s)
    return s


@pytest.mark.parametrize("entry", ENTRY_POINTS)
def test_cpu_tensors_are_rejected(entry):
    with pytest.raises(RuntimeError, match="CUDA-only"):
        ENTRY_POINTS[entry](_inputs("cpu"))


def test_host_forward_takes_a_dense_adjacency_only(spy):
    """The host-buffer entry points have no CSR form: a CSR triple or a CsrGraph is refused before the library."""
    d = _inputs("cpu")
    with pytest.raises(TypeError, match="adj_matrix must be a torch.Tensor"):
        ops.gcn_gru_forward_host(d["csr"], d["x"], d["params"], device=DEV)
    model = windgnn_b200.GCN_GRU(F, FH, F, S * F, H)
    with pytest.raises(TypeError, match="adj_matrix must be a torch.Tensor"):
        model.forward_host(windgnn_b200.CsrGraph(*d["csr"], S), d["x"])
    assert not [n for n in spy.names if n.startswith("wg_gcn_gru")]


@pytest.mark.gpu
def test_valid_inputs_run():
    d = _inputs(DEV)
    for entry in ("forward", "forward_csr"):
        assert ENTRY_POINTS[entry](d).shape == (2, 5, H)
    for entry in FORECASTS:
        assert ENTRY_POINTS[entry](d).shape == (2, H)
    assert ENTRY_POINTS["forward_host"](d).shape == (2, 5, H)
    assert ENTRY_POINTS["forward_train"](d)[0].shape == (2, 5, H)
    assert ENTRY_POINTS["backward"](d).numel() == sum(p.numel() for p in d["params"])
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ENTRY_POINTS)
def test_cpu_parameter_is_rejected(entry):
    d = _inputs(DEV)
    d["params"][2] = d["params"][2].cpu()
    with pytest.raises(RuntimeError, match="conv2.weight is on cpu; the fused path is CUDA-only"):
        ENTRY_POINTS[entry](d)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ENTRY_POINTS)
def test_float64_parameter_is_rejected(entry):
    d = _inputs(DEV)
    d["params"][5] = d["params"][5].double()
    with pytest.raises(RuntimeError, match="gru.weight_hh_l0 must be float32, got torch.float64"):
        ENTRY_POINTS[entry](d)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["conv1.weight", "conv2.bias", "gru.weight_ih_l0", "gru.weight_hh_l0"])
@pytest.mark.parametrize("entry", ENTRY_POINTS)
def test_parameter_of_the_wrong_shape_is_named(entry, name):
    d = _inputs(DEV)
    i = NAMES.index(name)
    shp = list(PARAMS[i][1])
    shp[0] += 1
    d["params"][i] = torch.zeros(shp, device=DEV)
    with pytest.raises(RuntimeError, match=name):
        ENTRY_POINTS[entry](d)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["forward", "forecast", "forward_host", "forward_train", "backward"])
def test_dense_adjacency_of_the_wrong_shape_is_rejected(entry):
    d = _inputs(DEV)
    d["adj"] = torch.full((S + 1, S + 1), 1.0 / S, device=DEV)
    with pytest.raises(RuntimeError, match=rf"adj_matrix must be \[{S}, {S}\]"):
        ENTRY_POINTS[entry](d)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", CSR_OPS)
def test_csr_arrays_are_checked(entry):
    d = _inputs(DEV)
    rowptr, colidx, vals = d["csr"]
    d["csr"] = (torch.cat([rowptr, rowptr[-1:]]), colidx, vals)
    with pytest.raises(RuntimeError, match="CSR arrays do not match the number of stations"):
        ENTRY_POINTS[entry](d)
    d["csr"] = (rowptr, colidx.long(), vals)
    with pytest.raises(RuntimeError, match="colidx must be a CUDA int32 tensor on cuda:0"):
        ENTRY_POINTS[entry](d)
    d["csr"] = (rowptr.cpu(), colidx, vals)
    with pytest.raises(RuntimeError, match="rowptr must be a CUDA int32 tensor on cuda:0"):
        ENTRY_POINTS[entry](d)
    d["csr"] = (rowptr, colidx, vals[:-1])
    with pytest.raises(RuntimeError, match="CSR arrays do not match the number of stations"):
        ENTRY_POINTS[entry](d)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", FORECASTS)
def test_forecast_starts_must_be_1d_int64(entry):
    d = _inputs(DEV)
    for bad in (d["starts"].int(), d["starts"][None]):
        d["starts"] = bad
        with pytest.raises(RuntimeError, match="starts must be a 1-D int64 tensor"):
            ENTRY_POINTS[entry](d)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(0, 5), (2, 0), (0, 0)])
@pytest.mark.parametrize("entry", ["forward", "forward_csr"])
def test_empty_forward_returns_without_calling_the_library(entry, B, T, spy):
    out = ENTRY_POINTS[entry](_inputs(DEV, B=B, T=T))
    assert out.shape == (B, T, H) and out.device == torch.device(DEV)
    assert not [n for n in spy.names if n.startswith("wg_gcn_gru")]


@pytest.mark.gpu
def test_empty_host_forward_returns_without_calling_the_library(spy):
    out = ENTRY_POINTS["forward_host"](_inputs(DEV, B=0))
    assert out.shape == (0, 5, H) and out.device.type == "cpu"
    assert not [n for n in spy.names if n.startswith("wg_gcn_gru")]


@pytest.mark.gpu
@pytest.mark.parametrize("entry", FORECASTS)
def test_forecast_without_windows_still_goes_to_the_library(entry, spy):
    entry_point = "wg_gcn_gru_forecast_csr_f32" if entry == "forecast_csr" else "wg_gcn_gru_forecast_f32"
    out = ENTRY_POINTS[entry](_inputs(DEV, n_starts=0))
    torch.cuda.synchronize()
    assert out.shape == (0, H) and entry_point in spy.names
    # the library still rejects a window longer than the table
    with pytest.raises(_lib.WindGNNError, match="L <= Ttot") as ei:
        ENTRY_POINTS[entry](_inputs(DEV, Ttot=L - 1, n_starts=0))
    assert ei.value.code == _lib.WG_ERR_BAD_ARG


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_host_forward_adjacency_must_be_on_the_device():
    d = _inputs(DEV)
    d["adj"] = d["adj"].to("cuda:1")
    with pytest.raises(RuntimeError, match="adj_matrix is on cuda:1, expected cuda:0"):
        ops.gcn_gru_forward_host(d["adj"], d["x"].cpu(), d["params"], device=DEV)
