"""GPU parity: the CUDA path (through the C-ABI) against the CPU oracle and against the committed
outputs of the unmodified reference module.  Tolerance: ``max|y - ref| / max|ref| <= 1e-5``
(BASELINE.json north_star, FP32 path; SURVEY.md 8(c) explains why the error is normalised)."""

import numpy as np
import pytest
import torch

import windgnn_b200
from conftest import golden, load_checkpoint
from oracle import gcn_gru_forward, gcn_layer, normalised_max_error
from windgnn_b200 import _lib, ops

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = "cuda:0"


def _model(S, sd=None):
    m = windgnn_b200.GCN_GRU(13, 13, 13, 13 * S, 3 * S)
    m.load_state_dict(sd if sd is not None else load_checkpoint(S), strict=True)
    return m.to(DEV).eval()


def _adj(S):
    return golden(f"adj_ref_{S}.npy").astype(np.float32)


@pytest.mark.parametrize("S", [7, 34])
def test_forward_matches_reference_golden_and_oracle(S):
    g = golden(f"fwd_{S}.npz")
    adj = _adj(S)
    model = _model(S)
    with torch.no_grad():
        y = model(torch.from_numpy(adj).to(DEV), torch.from_numpy(g["x"]).to(DEV)).cpu().numpy()
    assert y.shape == g["y_ref_f32"].shape
    assert np.isfinite(y).all()
    assert normalised_max_error(y, g["y_ref_f32"]) <= TOL           # the reference module, fp32
    assert normalised_max_error(y, g["y_ref_f64"]) <= TOL           # fp64 ground truth
    ref = gcn_gru_forward(adj, g["x"], load_checkpoint(S), dtype=np.float32)
    assert normalised_max_error(y, ref) <= TOL                      # the oracle


@pytest.mark.parametrize("S", [7, 34])
def test_batch_one_returns_T_by_H_like_the_reference(S):
    g = golden(f"fwd_{S}.npz")
    model = _model(S)
    adj = torch.from_numpy(_adj(S)).to(DEV)
    with torch.no_grad():
        y = model(adj, torch.from_numpy(g["x"][1:2]).to(DEV))       # [1, T, S, 13] — main.py:102
    assert y.shape == (168, 3 * S)                                  # squeeze(0), step6:26
    assert normalised_max_error(y.cpu().numpy(), g["y_ref_f32"][1]) <= TOL


def test_short_windows():
    g = golden("fwd_34_short.npz")
    model = _model(34)
    adj = torch.from_numpy(_adj(34)).to(DEV)
    for T in (1, 5):
        with torch.no_grad():
            y = model(adj, torch.from_numpy(g[f"x_T{T}"]).to(DEV)).cpu().numpy()
        assert y.shape == (T, 102)
        assert normalised_max_error(y, g[f"y_T{T}"][0]) <= TOL


def test_non_default_dims_generic_kernels():
    """GCN_GRU(6, 10, 13, 65, 11) on S = 5: F_in != F_hid != 13, H != 3S."""
    g = golden("fwd_rand.npz")
    params = {k.replace("__", "."): torch.from_numpy(g[k]) for k in g.files if "__" in k}
    m = windgnn_b200.GCN_GRU(6, 10, 13, 65, 11)
    m.load_state_dict(params, strict=True)
    m = m.to(DEV).eval()
    with torch.no_grad():
        y = m(torch.from_numpy(g["adj"]).to(DEV), torch.from_numpy(g["x"]).to(DEV)).cpu().numpy()
    assert y.shape == (4, 9, 11)
    assert normalised_max_error(y, g["y_ref_f32"]) <= TOL


@pytest.mark.parametrize("dims", [(3, 5, 13, 13), (37, 34, 13, 13), (2, 9, 6, 10), (1, 40, 16, 3)])
def test_gcn_layer_op(dims):
    R, S, Fi, Fo = dims
    rng = np.random.default_rng(R * 1000 + S)
    adj = rng.random((S, S), dtype=np.float32) / S
    attr = rng.random((R, 3, S, Fi), dtype=np.float32)              # extra leading dims like [B, T, S, F]
    w = rng.standard_normal((Fi, Fo)).astype(np.float32)
    b = rng.standard_normal(Fo).astype(np.float32)
    layer = windgnn_b200.GraphConvLayer(Fi, Fo)
    layer.load_state_dict({"weight": torch.from_numpy(w), "bias": torch.from_numpy(b)})
    layer = layer.to(DEV)
    with torch.no_grad():
        y = layer(torch.from_numpy(adj).to(DEV), torch.from_numpy(attr).to(DEV)).cpu().numpy()
    ref = gcn_layer(adj, attr, w, b)
    assert y.shape == ref.shape
    assert normalised_max_error(y, ref) <= TOL
    assert (y >= 0).all()


def _random_model(S, seed, H=None):
    torch.manual_seed(seed)
    H = H or 3 * S
    m = windgnn_b200.GCN_GRU(13, 13, 13, 13 * S, H)
    with torch.no_grad():
        m.conv1.weight.mul_(0.3)
        m.conv2.weight.mul_(0.3)
    return m


@pytest.mark.parametrize("S,H,B,T", [(1, 3, 5, 4), (3, 9, 33, 7), (12, 36, 70, 11), (34, 102, 65, 9), (20, 50, 31, 6),
                                     (33, 99, 37, 5)])
def test_ragged_shapes_vs_oracle(S, H, B, T):
    """Batch sizes that are not multiples of the 32-sequence CTA tile, odd S / H, row tiles cut by
    the end of the batch."""
    m = _random_model(S, seed=S * 100 + B, H=H)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    rng = np.random.default_rng(B)
    adj = (rng.random((S, S), dtype=np.float32) / S).astype(np.float32)
    x = rng.random((B, T, S, 13), dtype=np.float32)
    ref = gcn_gru_forward(adj, x, sd, dtype=np.float32)
    with torch.no_grad():
        y = m.to(DEV)(torch.from_numpy(adj).to(DEV), torch.from_numpy(x).to(DEV))
    y = y.reshape(B, T, H).cpu().numpy()
    assert normalised_max_error(y, ref) <= TOL


@pytest.mark.parametrize("S,B,T", [(34, 70, 6), (33, 45, 4), (31, 40, 3)])
def test_gcn_generations_are_bit_identical(S, B, T, monkeypatch):
    """gcn_rows_kernel (S = 33 / 34: four station pairs per warp plus a feature slice of the shared 17th pair;
    S = 31: the uneven split) against the first-generation gcn_kernel: every sum keeps its order."""
    m = _random_model(S, seed=S + B).to(DEV)
    rng = np.random.default_rng(S * 31 + B)
    adj = torch.from_numpy((rng.random((S, S), dtype=np.float32) / S).astype(np.float32)).to(DEV)
    x = torch.from_numpy(rng.random((B, T, S, 13), dtype=np.float32) - 0.25).to(DEV)
    with torch.no_grad():
        monkeypatch.setenv("WG_FORCE_LEGACY", "1")
        y_old = m(adj, x)
        monkeypatch.setenv("WG_FORCE_LEGACY", "0")
        y_new = m(adj, x)
    assert torch.equal(y_old, y_new)


def test_empty_batch():
    m = _model(7)
    y = m(torch.from_numpy(_adj(7)).to(DEV), torch.zeros((0, 168, 7, 13), device=DEV))
    assert y.shape == (0, 168, 21)


# ---------------------------------------------------------------------------------------------
# size-independent properties at BASELINE.json's full size (config[1]: S = 34, B = 4096, T = 168)
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def full34():
    model = _model(34)
    adj = torch.from_numpy(_adj(34)).to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(0)
    x = torch.rand((4096, 168, 34, 13), generator=gen, device=DEV)
    with torch.no_grad():
        y = model(adj, x)
    torch.cuda.synchronize()
    return model, adj, x, y


def test_full_size_sample_vs_oracle(full34):
    model, adj, x, y = full34
    assert y.shape == (4096, 168, 102) and torch.isfinite(y).all()
    idx = [0, 31, 32, 2047, 4064, 4095]                               # first/last of CTA tiles
    ref = gcn_gru_forward(adj.cpu().numpy(), x[idx].cpu().numpy(), load_checkpoint(34))
    assert normalised_max_error(y[idx].cpu().numpy(), ref) <= TOL


def test_full_size_chunking_and_sharding_invariance(full34):
    """Sequences are independent: any split of the batch (internal chunks, or the per-GPU shards of
    the multi-GPU run) gives bit-identical results."""
    model, adj, x, y = full34
    with torch.no_grad():
        model.chunk = 1000                                            # ragged internal chunks
        y_chunked = model(adj, x)
        model.chunk = 0
        shards = [model(adj, x[lo:hi]) for lo, hi in ((0, 512), (512, 1024), (1024, 4096))]
    assert torch.equal(y_chunked, y)
    assert torch.equal(torch.cat(shards), y)


def test_small_batch_recurrence_is_bit_identical_to_the_throughput_kernel(full34):
    """Up to 1,184 sequences the 4-sequence-per-CTA recurrence (gru_recur_regw_kernel) runs, above that
    gru_recur_unit_kernel: same summation order, same gate expressions -> the same bits, for a single
    window (the reference's batch-1 call, main.py:102), ragged CTAs and the 7-station model."""
    model, adj, x, y = full34
    with torch.no_grad():
        for lo, hi in ((0, 1), (5, 8), (100, 703), (2000, 3184), (2000, 3185)):
            assert torch.equal(model(adj, x[lo:hi]).reshape(hi - lo, 168, 102), y[lo:hi]), (lo, hi)
    m7 = _model(7)
    adj7 = torch.from_numpy(_adj(7)).to(DEV)
    x7 = torch.rand((1300, 24, 7, 13), device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    with torch.no_grad():
        big = m7(adj7, x7)                                            # 1300 > 1184: throughput kernel
        small = torch.cat([m7(adj7, x7[:650]), m7(adj7, x7[650:])])   # 650 each: small-batch kernel
    assert torch.equal(big, small)


def test_full_size_determinism_and_permutation(full34):
    model, adj, x, y = full34
    perm = torch.randperm(512, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
    with torch.no_grad():
        y2 = model(adj, x[:512])
        yp = model(adj, x[:512][perm])
    assert torch.equal(y2, y[:512])                                   # idempotent / deterministic
    assert torch.equal(yp, y[:512][perm])                             # permutation equivariant


def test_full_size_causality(full34):
    """h_t depends on x_0..x_t only: the forward of a truncated window is a prefix."""
    model, adj, x, y = full34
    with torch.no_grad():
        y_short = model(adj, x[:64, :50].contiguous())
    assert torch.equal(y_short, y[:64, :50])
    assert y.abs().max() < 1.0                                        # GRU states live in (-1, 1)


def test_host_buffer_path_matches_device_path(full34):
    model, adj, x, y = full34
    xh = x[:1500].cpu().pin_memory()
    model.chunk = 400
    try:
        out = model.forward_host(adj, xh)
    finally:
        model.chunk = 0
    assert out.shape == (1500, 168, 102) and not out.is_cuda
    assert torch.equal(out, y[:1500].cpu())
    # second call on the same thread reuses the cached internal streams / events
    assert torch.equal(model.forward_host(adj, xh), out)


def test_host_predict_returns_only_the_denormalised_last_step(full34):
    """wg_gcn_gru_predict_host_f32: the evaluation loop of main.py:101-116 in one call — only 3S floats per
    window come back; bit-identical to the full host forward followed by the library's de-normalisation."""
    model, adj, x, y = full34
    xh = x[:700].cpu().pin_memory()
    wmin, wmax = 0.0, 83.6
    pred = model.forward_host(adj, xh, last_step_range=(wmin, wmax))
    assert pred.shape == (700, 102) and not pred.is_cuda
    ref = windgnn_b200.denormalise_last_step(y[:700], wmin, wmax).cpu()
    assert torch.equal(pred, ref)


def test_stage_entry_points_compose(full34):
    """The three stage entry points chained by hand equal the fused call."""
    model, adj, x, y = full34
    lib = _lib.load()
    B, dims = 256, (168, 34, 13, 13, 13, 102)
    nbytes = lib.wg_gcn_gru_workspace_bytes(B, *dims, B, 0)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    out = torch.empty((B, 168, 102), device=DEV)
    p = [t.detach().contiguous() for t in (
        model.conv1.weight, model.conv1.bias, model.conv2.weight, model.conv2.bias,
        model.gru.weight_ih_l0, model.gru.weight_hh_l0, model.gru.bias_ih_l0, model.gru.bias_hh_l0)]
    st = torch.cuda.current_stream().cuda_stream
    xs = x[:B].contiguous()
    _lib.check(lib.wg_stage_pack_f32(*(t.data_ptr() for t in p[4:]), *dims, B, 0, ws.data_ptr(), nbytes, 0, st))
    _lib.check(lib.wg_stage_gcn_f32(adj.data_ptr(), xs.data_ptr(), *(t.data_ptr() for t in p[:4]), B, *dims, B, 0,
                                    ws.data_ptr(), nbytes, 0, st))
    _lib.check(lib.wg_stage_inproj_f32(B, *dims, B, 0, ws.data_ptr(), nbytes, 0, st))
    _lib.check(lib.wg_stage_recur_f32(out.data_ptr(), B, *dims, B, 0, ws.data_ptr(), nbytes, 0, st))
    torch.cuda.synchronize()
    assert torch.equal(out, y[:B])


# ---------------------------------------------------------------------------------------------
# tensor-core path: GRU input projection on tcgen05 with error-compensated TF32 (3xTF32).
# Stated tolerance: the SAME 1e-5 normalised bar as the FP32 path (three TF32 products per term
# reproduce fp32 products to ~2^-21, fp32 accumulate).
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [7, 34])
def test_tensor_core_path_matches_reference_golden(S):
    g = golden(f"fwd_{S}.npz")
    model = _model(S)
    model.precision = "tf32x3"
    adj = torch.from_numpy(_adj(S)).to(DEV)
    with torch.no_grad():
        y = model(adj, torch.from_numpy(g["x"]).to(DEV)).cpu().numpy()
    assert np.isfinite(y).all()
    assert normalised_max_error(y, g["y_ref_f32"]) <= TOL
    assert normalised_max_error(y, g["y_ref_f64"]) <= TOL


def test_tensor_core_path_full_size(full34):
    model, adj, x, y = full34
    model.precision = "tf32x3"
    try:
        with torch.no_grad():
            yt = model(adj, x)
            yt2 = model(adj, x[1000:1300])
    finally:
        model.precision = "fp32"
    torch.cuda.synchronize()
    # against the FP32-FMA path on all 4096 sequences, and shard invariance of the tensor path itself
    err = float((yt - y).abs().max() / y.abs().max())
    assert err <= TOL, err
    assert torch.equal(yt2, yt[1000:1300])
    idx = [0, 127, 128, 4095]
    ref = gcn_gru_forward(adj.cpu().numpy(), x[idx].cpu().numpy(), load_checkpoint(34))
    assert normalised_max_error(yt[idx].cpu().numpy(), ref) <= TOL


@pytest.mark.parametrize("S,H,B,T", [(3, 9, 33, 7), (12, 36, 70, 11), (20, 50, 31, 6), (40, 150, 9, 5)])
def test_tensor_core_path_ragged_shapes(S, H, B, T):
    m = _random_model(S, seed=S * 7 + B, H=H)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    rng = np.random.default_rng(B + 1)
    adj = (rng.random((S, S), dtype=np.float32) / S).astype(np.float32)
    x = rng.random((B, T, S, 13), dtype=np.float32)
    ref = gcn_gru_forward(adj, x, sd, dtype=np.float32)
    m = m.to(DEV)
    m.precision = "tf32x3"
    with torch.no_grad():
        y = m(torch.from_numpy(adj).to(DEV), torch.from_numpy(x).to(DEV)).reshape(B, T, H).cpu().numpy()
    assert normalised_max_error(y, ref) <= TOL


def _scaled_model(S, Fh, H, seed):
    """GCN_GRU(13, Fh, 13, 13*S, H) with the weight scale SURVEY.md 8(d) prescribes for wide layers
    (unscaled randn saturates the GRU)."""
    torch.manual_seed(seed)
    m = windgnn_b200.GCN_GRU(13, Fh, 13, 13 * S, H)
    with torch.no_grad():
        m.conv1.weight.mul_(0.05)
        m.conv2.weight.mul_(0.05)
    return m


@pytest.mark.parametrize("S,Fh,H,B,T,k", [(300, 128, 128, 3, 6, 8), (96, 40, 30, 5, 4, 3), (150, 13, 36, 2, 5, 8),
                                           (300, 320, 48, 2, 3, 8), (4600, 16, 32, 1, 2, 4)])
def test_sparse_graph_path_vs_oracle(S, Fh, H, B, T, k):
    """CSR adjacency path (large kNN graph, wide GCN hidden layer) against the oracle.  The last two cases run
    gcn_sparse_l1_kernel / gcn_sparse_l2_kernel: F_hid = 320 is wider than the constant bank of
    gcn_sparse_plan_kernel, and a 4600-station slab does not fit shared memory."""
    from oracle import knn_graph_f64, synthetic_coordinates

    adj = knn_graph_f64(synthetic_coordinates(S, seed=S), k).astype(np.float32)
    m = _scaled_model(S, Fh, H, seed=S + B)
    sd = {kk: v.detach().clone() for kk, v in m.state_dict().items()}
    x = np.random.default_rng(S).random((B, T, S, 13), dtype=np.float32)
    ref = gcn_gru_forward(adj, x, sd, dtype=np.float32)
    m = m.to(DEV)
    m.DENSE_MAX_STATIONS = 64                                          # force the CSR path for S = 96 too
    with torch.no_grad():
        y = m(torch.from_numpy(adj).to(DEV), torch.from_numpy(x).to(DEV)).reshape(B, T, H).cpu().numpy()
    assert normalised_max_error(y, ref) <= TOL


def test_sparse_path_matches_reference_class_golden_at_wide_dims():
    """fwd_wide.npz was made by the unmodified reference CLASS, GCN_GRU(13, 128, 13, 3900, 128), on a 300-station
    kNN graph (tests/golden/make_golden.py).  The CSR kernels evaluate layer 2 as A.(G1.W2) instead of the
    reference's (A.G1).W2: this is the fixture that pins that re-association to the reference itself."""
    g = golden("fwd_wide.npz")
    S, Fh, H = 300, 128, 128
    m = windgnn_b200.GCN_GRU(13, Fh, 13, 13 * S, H)
    m.load_state_dict({k.replace("__", "."): torch.from_numpy(g[k]) for k in g.files if "__" in k}, strict=True)
    m = m.to(DEV).eval()
    with torch.no_grad():
        y = m(torch.from_numpy(g["adj"]).to(DEV), torch.from_numpy(g["x"]).to(DEV)).cpu().numpy()
    assert y.shape == g["y_ref_f32"].shape == (2, 6, H)
    assert normalised_max_error(y, g["y_ref_f32"]) <= TOL
    assert normalised_max_error(y, g["y_ref_f64"]) <= TOL
    # the oracle agrees with the same fixture (so the oracle-only checks of configs[3] rest on the reference too)
    sd = {k.replace("__", "."): g[k] for k in g.files if "__" in k}
    assert normalised_max_error(gcn_gru_forward(g["adj"], g["x"], sd, dtype=np.float32), g["y_ref_f32"]) <= 3e-6


def test_config4_4096_station_knn_graph():
    """BASELINE.json configs[3]: synthetic 4096-station kNN(k=8) graph, GCN hidden 128, 24-step window
    (GRU hidden 128 — SURVEY.md 8(d) variant C), graph built on the GPU, forward against the oracle."""
    S, Fh, H, B, T = 4096, 128, 128, 2, 24
    latlon = windgnn_b200.synthetic_coordinates(S, seed=0, device=DEV).cpu().numpy()
    adj = windgnn_b200.knn_graph_from_latlon(latlon, k=8, device=DEV)
    assert int((adj != 0).sum(1).max()) < 64
    m = _scaled_model(S, Fh, H, seed=4)
    sd = {kk: v.detach().clone() for kk, v in m.state_dict().items()}
    x = np.random.default_rng(0).random((B, T, S, 13), dtype=np.float32)
    ref = gcn_gru_forward(adj.cpu().numpy(), x, sd, dtype=np.float32)
    with torch.no_grad():
        y = m.to(DEV)(adj, torch.from_numpy(x).to(DEV)).cpu().numpy()
    assert y.shape == (B, T, H)
    assert normalised_max_error(y, ref) <= TOL
    # shard / chunk invariance holds on this path too
    with torch.no_grad():
        y1 = m(adj, torch.from_numpy(x[1:]).to(DEV)).cpu().numpy()
    assert np.array_equal(y1, y[1])


def test_errors_are_reported_not_thrown_across_the_abi():
    m = windgnn_b200.GCN_GRU(20, 20, 13, 13 * 4, 12).to(DEV)          # F_in 20 > 16: unsupported on both paths
    with pytest.raises(_lib.WindGNNError) as ei:
        m(torch.eye(4, device=DEV), torch.zeros((2, 3, 4, 20), device=DEV))
    assert ei.value.code == _lib.WG_ERR_UNSUPPORTED
    # the code is the library's own, whichever limit the shape exceeds; planning rejects both, so nothing launches
    S = 80700   # S * F_out = 1,049,100 > 2^20
    eye = torch.arange(S + 1, dtype=torch.int32, device=DEV)
    params = [torch.zeros(shp, device=DEV) for shp in ((13, 13), (13,), (13, 13), (13,), (3, S * 13), (3, 1), (3,), (3,))]
    with pytest.raises(_lib.WindGNNError) as ei:
        ops.gcn_gru_forward_csr(eye, eye[:S], torch.ones(S, device=DEV), torch.zeros((1, 1, S, 13), device=DEV),
                                *params)
    assert ei.value.code == _lib.WG_ERR_UNSUPPORTED and "dimension too large" in str(ei.value)
    H = 400     # the wide recurrence's state does not fit shared memory
    params = [torch.zeros(shp, device=DEV) for shp in ((13, 13), (13,), (13, 13), (13,), (3 * H, 4 * 13), (3 * H, H),
                                                        (3 * H,), (3 * H,))]
    with pytest.raises(_lib.WindGNNError) as ei:
        ops.gcn_gru_forward_host(torch.eye(4, device=DEV), torch.zeros((2, 3, 4, 13)), params)
    assert ei.value.code == _lib.WG_ERR_UNSUPPORTED and f"GRU hidden size {H}" in str(ei.value)
    bad = _model(7)
    with pytest.raises(RuntimeError):
        bad(torch.eye(7, device=DEV), torch.zeros((2, 3, 9, 13), device=DEV))   # S mismatch


def test_ffma_peak_probe():
    t = _lib.load().wg_measure_ffma_tflops(0, 5)
    assert 20.0 < t < 100.0   # B200: 148 SM x 128 FFMA/clk x 2 x ~1.9 GHz ~ 72
