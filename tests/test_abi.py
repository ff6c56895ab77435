"""CPU-side checks of the C-ABI library: it loads, exports every symbol the header declares,
and its host logic (planning, validation, error reporting) behaves.  No compute calls."""

import ctypes
import os
import re

import pytest

from conftest import ROOT
from windgnn_b200 import _lib

HEADER = os.path.join(ROOT, "include", "windgnn_b200.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(wg_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_loads():
    from windgnn_b200 import build

    path = build.build()
    assert os.path.exists(path)
    lib = _lib.load()
    assert lib.wg_abi_version() == _lib.ABI_VERSION == 4


def test_every_declared_symbol_is_exported():
    names = declared_symbols()
    assert len(names) >= 14
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} declared in the header but not exported"
    # the Python binding types exactly the declared set
    assert sorted(_lib.exported_names()) == names


def test_workspace_planning():
    lib = _lib.load()
    dims34 = (168, 34, 13, 13, 13, 102)
    one = lib.wg_gcn_gru_workspace_bytes(1, *dims34, 0, 0)
    big = lib.wg_gcn_gru_workspace_bytes(4096, *dims34, 0, 0)
    assert 0 < one < big
    # scratch per sequence = T * (IP + GP) * 4 with IP = 448, GP = 312 (U is kept in 128-row tiles)
    per_seq = (big - lib.wg_gcn_gru_workspace_bytes(4096 - 128, *dims34, 0, 0)) / 128
    assert per_seq == pytest.approx(168 * (448 + 312) * 4, rel=1e-3)
    # the default chunk caps the scratch: 1M sequences need no more than one wave's worth
    assert lib.wg_gcn_gru_workspace_bytes(1 << 20, *dims34, 0, 0) == lib.wg_gcn_gru_workspace_bytes(148 * 32, *dims34, 0, 0)
    assert lib.wg_gcn_gru_workspace_bytes(1 << 20, *dims34, 1024, 0) < big
    # host-buffer path: two compute lanes + three staging slots each for x and out; chunk 0 = pieces of 256
    assert lib.wg_gcn_gru_host_workspace_bytes(4096, *dims34, 4096, 0) > 2 * big
    assert lib.wg_gcn_gru_host_workspace_bytes(4096, *dims34, 0, 0) == lib.wg_gcn_gru_host_workspace_bytes(4096, *dims34, 256, 0)
    assert lib.wg_gcn_gru_host_workspace_bytes(4096, *dims34, 0, 0) < big
    # the tensor-core path reads the same fp32 U tiles (no hi / lo copies in HBM): its scratch differs only by
    # the packed fp16 weights; unknown flags are rejected
    tc = lib.wg_gcn_gru_workspace_bytes(4096, *dims34, 0, _lib.FLAG_TENSOR_CORES)
    assert 0 < abs(tc - big) < 4 << 20
    assert lib.wg_gcn_gru_csr_workspace_bytes(256, 24, 4096, 13, 128, 13, 128, 0, _lib.FLAG_TENSOR_CORES) > 0
    assert lib.wg_build_graph_csr_workspace_bytes(4096, 8) < lib.wg_build_graph_workspace_bytes(4096, 8) // 20
    assert lib.wg_gcn_gru_workspace_bytes(4096, *dims34, 0, 8) == 0
    assert lib.wg_gcn_gru_workspace_bytes(8, 0, 34, 13, 13, 13, 102, 0, 0) == 0  # T = 0 is invalid
    assert "non-positive" in _lib.last_error()
    assert lib.wg_build_graph_workspace_bytes(34, 0) >= 34 * 34 * 8
    assert lib.wg_build_graph_workspace_bytes(4096, 8) > lib.wg_build_graph_workspace_bytes(4096, 0)


def test_argument_validation_happens_before_cuda():
    lib = _lib.load()
    dims = (4, 7, 13, 13, 13, 21)
    rc = lib.wg_gcn_gru_forward_f32(*([None] * 11), -1, *dims, 0, 0, None, 0, 0, None)
    assert rc == _lib.WG_ERR_BAD_ARG
    rc = lib.wg_gcn_gru_forward_f32(*([None] * 11), 2, *dims, 0, 0, None, 0, 0, None)
    assert rc == _lib.WG_ERR_BAD_ARG and "null" in _lib.last_error()
    # B == 0 is a valid no-op
    assert lib.wg_gcn_gru_forward_f32(*([None] * 11), 0, *dims, 0, 0, None, 0, 0, None) == _lib.WG_OK
    rc = lib.wg_gcn_layer_f32(None, None, None, None, None, 3, 7, 13, 13, 0, None)
    assert rc == _lib.WG_ERR_BAD_ARG
    with pytest.raises(_lib.WindGNNError):
        _lib.check(rc)
    # misaligned / short workspace is rejected with its own code
    buf = ctypes.create_string_buffer(1024)
    addr = (ctypes.addressof(buf) + 255) // 256 * 256
    fake = ctypes.c_void_p(8)  # non-null, never dereferenced: validation fails first
    rc = lib.wg_gcn_gru_forward_f32(*([fake] * 11), 2, *dims, 0, 0, ctypes.c_void_p(addr), 16, 0, None)
    assert rc == _lib.WG_ERR_WORKSPACE and "too small" in _lib.last_error()
    rc = lib.wg_gcn_gru_forward_f32(*([fake] * 11), 2, *dims, 0, 0, ctypes.c_void_p(addr + 4), 1 << 30, 0, None)
    assert rc == _lib.WG_ERR_WORKSPACE and "aligned" in _lib.last_error()


@pytest.mark.parametrize("csr,dims,reason", [
    (False, (4, 168, 7, 20, 20, 13, 21, 0, 0), "GCN feature width 20 > 16"),
    (False, (4, 8, 520, 16, 16, 16, 21, 0, 0), "S=520 too large for the dense GCN kernel"),
    (False, (4, 8, 600, 13, 13, 13, 21, 0, 0), "S=600 too large for the dense GCN kernel"),   # the 13 x 4 kernel
    (False, (4, 8, 200, 16, 16, 16, 21, 0, 0), "dense GCN needs"),
    (False, (4, 8, 34, 13, 13, 13, 400, 0, 0), "GRU hidden size 400: state does not fit"),
    (True, (2, 3, 4, 20, 20, 13, 12, 0, 0), "sparse GCN: F_in / F_out must be <= 16 (got 20 / 13)"),
    (True, (2, 3, 300, 13, 2000, 13, 24, 0, 0), "sparse GCN: hidden width 2000 too large"),
    (True, (20000, 168, 300, 13, 32, 13, 24, 20000, 0), "sparse GCN: chunk of 3360000 rows too large"),
    (True, (2, 3, 300, 13, 32, 13, 400, 0, 0), "GRU hidden size 400: state does not fit"),
])
def test_kernel_limits_are_checked_at_planning(csr, dims, reason):
    """A shape that no kernel of the plan serves gets no workspace, and the forward rejects it before it looks at the
    workspace, so that nothing launches."""
    lib = _lib.load()
    query, entry, n_ptrs = ((lib.wg_gcn_gru_csr_workspace_bytes, lib.wg_gcn_gru_forward_csr_f32, 13) if csr else
                            (lib.wg_gcn_gru_workspace_bytes, lib.wg_gcn_gru_forward_f32, 11))
    assert query(*dims) == 0
    assert reason in _lib.last_error()
    fake = ctypes.c_void_p(8)   # non-null, never dereferenced; the workspace stays NULL so that nothing can launch
    assert entry(*([fake] * n_ptrs), *dims, None, 0, 0, None) == _lib.WG_ERR_UNSUPPORTED
    assert reason in _lib.last_error()


def test_training_planning_and_validation():
    lib = _lib.load()
    dims34 = (168, 34, 13, 13, 13, 102)
    n34 = 13 * 13 + 13 + 13 * 13 + 13 + 306 * 442 + 306 * 102 + 306 + 306
    assert lib.wg_gcn_gru_param_count(34, 13, 13, 13, 102) == n34 == 167440     # SURVEY.md 8(a) row C
    assert lib.wg_gcn_gru_param_count(7, 13, 13, 13, 21) == 7546
    fwd = lib.wg_gcn_gru_workspace_bytes(512, *dims34, 512, 0)
    trn = lib.wg_gcn_gru_train_workspace_bytes(512, *dims34)
    # saved gates + DG (4H each) + dU (I) per row on top of the forward's scratch
    assert trn - fwd >= 512 * 168 * (2 * 408 + 442) * 4
    assert lib.wg_gcn_gru_train_workspace_bytes(512, 168, 34, 13, 32, 13, 102) == 0
    assert "feature widths" in _lib.last_error()
    # the training limits are reported before the forward's, which these shapes exceed too
    assert lib.wg_gcn_gru_train_workspace_bytes(4, 8, 520, 16, 16, 16, 21) == 0
    assert _lib.last_error() == "training: S=520 too large for the dense GCN kernels"
    assert lib.wg_gcn_gru_train_workspace_bytes(4, 8, 200, 16, 16, 16, 21) == 0
    assert _lib.last_error() == "training: S=200 does not fit the shared-memory GCN backward"
    assert lib.wg_mse_workspace_bytes() >= 8
    fake = ctypes.c_void_p(8)
    rc = lib.wg_gcn_gru_forward_train_f32(*([fake] * 11), 2, *dims34, None, 0, 0, None)
    assert rc == _lib.WG_ERR_WORKSPACE
    rc = lib.wg_gcn_gru_backward_f32(*([None] * 11), 2, *dims34, None, 0, 0, None)
    assert rc == _lib.WG_ERR_BAD_ARG and "null" in _lib.last_error()
    # B*T is bounded by the one-pass dU stage: 12482 x 168 rows plan, 12483 x 168 are rejected before any launch
    assert lib.wg_gcn_gru_train_workspace_bytes(12482, *dims34) > 0
    assert lib.wg_gcn_gru_train_workspace_bytes(12483, *dims34) == 0
    assert "rows" in _lib.last_error()
    rc = lib.wg_gcn_gru_forward_train_f32(*([fake] * 11), 12483, *dims34, None, 0, 0, None)
    assert rc == _lib.WG_ERR_UNSUPPORTED and "rows" in _lib.last_error()
    rc = lib.wg_gcn_gru_backward_f32(*([fake] * 11), 12483, *dims34, None, 0, 0, None)
    assert rc == _lib.WG_ERR_UNSUPPORTED and "rows" in _lib.last_error()
    assert lib.wg_mse_loss_grad_f32(None, None, 0, None, None, None, 0, 0, None) == _lib.WG_ERR_BAD_ARG
    assert lib.wg_adam_step_f32(None, None, None, None, 10, 1e-3, 0.9, 0.999, 1e-8, 0, 1.0, 0, None) == _lib.WG_ERR_BAD_ARG
    assert lib.wg_adam_step_f32(None, None, None, None, 0, 1e-3, 0.9, 0.999, 1e-8, 1, 1.0, 0, None) == _lib.WG_OK


def test_integration_doc_binding_matches_the_library():
    """INTEGRATION.md section 3 is the binding a maintainer copies: execute it against the built library
    and compare what it declares with the typed binding the package itself uses (ABI v3: `flags`
    after `chunk` in both calls)."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    sec = text[text.index("## 3. Raw ctypes binding"):text.index("## 4. Contract")]
    code = re.search(r"```python\n(.*?)```", sec, flags=re.S).group(1)
    ns = {}
    cwd = os.getcwd()
    os.chdir(ROOT)   # the snippet opens the library by its in-tree relative path
    try:
        exec(compile(code, "INTEGRATION.md#3", "exec"), ns)
    finally:
        os.chdir(cwd)
    doc = ns["lib"]
    for name in ("wg_gcn_gru_workspace_bytes", "wg_gcn_gru_forward_f32"):
        restype, argtypes = _lib._SIGNATURES[name]
        fn = getattr(doc, name)
        assert fn.restype is restype
        assert [ctypes.sizeof(a) for a in fn.argtypes] == [ctypes.sizeof(a) for a in argtypes]
        assert len(fn.argtypes) == len(argtypes)
    dims34 = (168, 34, 13, 13, 13, 102)
    # the documented call and the package's typed call plan the same workspace, for both flag values
    for flags in (0, ns["WG_FLAG_TENSOR_CORES"]):
        assert doc.wg_gcn_gru_workspace_bytes(4096, *dims34, 0, flags) == \
            _lib.load().wg_gcn_gru_workspace_bytes(4096, *dims34, 0, flags) > 0
    # argument validation through the documented signature: a short workspace is rejected as such
    fake = ctypes.c_void_p(256)
    rc = doc.wg_gcn_gru_forward_f32(*([fake] * 11), 2, *dims34, 0, 0, fake, 16, 0, None)
    assert rc == _lib.WG_ERR_WORKSPACE and b"too small" in doc.wg_last_error()
    assert callable(ns["gcn_gru_forward"])
