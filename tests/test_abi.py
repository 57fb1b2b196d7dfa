"""C-ABI surface: the library loads and exports every symbol include/dva_b200.h declares.
No compute is launched here (argument validation only), so this runs without a GPU."""
import ctypes
import os
import re

import pytest

from conftest import ROOT
from deepviewagg_b200 import _lib


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "dva_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dva_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_all_exported():
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/dva_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature in _lib.py"
    assert set(_lib.SIGNATURES) == set(names)


def test_abi_version_and_error_string():
    lib = _lib.load()
    assert lib.dva_abi_version() == 1
    # negative size -> DVA_EINVAL before anything is launched
    rc = lib.dva_segment_csr_fwd(None, None, None, None, -1, 0, 4, 0, 0, None)
    assert rc == _lib.DVA_EINVAL
    assert b"segment_csr_fwd" in lib.dva_last_error()
    # G not a power of two -> DVA_EUNSUPPORTED (host composes the unfused operators then)
    rc = lib.dva_view_attention_fwd(None, None, 0, None, None, None, None, None, None, None, None,
                                    None, 4, 4, 4, 12, 3, 0, 1e-12, 0, None)
    assert rc == _lib.DVA_EUNSUPPORTED
    rc = lib.dva_view_attention_fwd(None, None, 0, None, None, None, None, None, None, None, None,
                                    None, 4, 4, 4, 2, 4, 0, 1e-12, 0, None)
    assert rc == _lib.DVA_EINVAL  # more groups than channels
    assert lib.dva_view_attention_bwd_workspace_bytes(4) > 0


def test_knobs_and_workspace_queries_validate_arguments():
    lib = _lib.load()
    # kernels of the fused pair: 0 auto, 1 streaming, 2 ring fwd + lane bwd, 3 streaming fwd + lane bwd; anything else is refused
    assert lib.dva_view_attention_set_path(4) == _lib.DVA_EINVAL
    assert lib.dva_view_attention_set_path(-1) == _lib.DVA_EINVAL
    for path in (1, 2, 3, 0):
        assert lib.dva_view_attention_set_path(path) == 0
    # projection workspace: narrow layers (K, N <= 64) are served by the skinny kernels for any K / N;
    # only dW (layout 2) needs room for the per-CTA partials
    assert lib.dva_linear_gemm_workspace_bytes(100000, 32, 33, 0, 0) >= 16
    small = lib.dva_linear_gemm_workspace_bytes(100000, 32, 33, 2, 0)
    assert small >= 32 * 33 * 4
    # wide layers need 16-byte rows for TMA: K % 4 != 0 has no workspace (ops.linear zero-pads such widths)
    assert lib.dva_linear_gemm_workspace_bytes(1000, 128, 132, 0, 0) > 0
    assert lib.dva_linear_gemm_workspace_bytes(1000, 128, 131, 0, 0) == 0
    rc = lib.dva_linear_gemm(None, None, None, 10, 128, 131, 0, 0, None, 0, None)
    assert rc == _lib.DVA_EUNSUPPORTED


def test_mlp_layer_entry_points_validate_shapes():
    """Host-side shape rules of the fused layer entry points (no launch)."""
    lib = _lib.load()
    # fused narrow-layer backward: N <= 32 outputs, K <= 64 inputs, both multiples of 4
    assert lib.dva_mlp_layer_bwd_supported(1000, 32, 32) == 1
    assert lib.dva_mlp_layer_bwd_supported(1000, 32, 8) == 1
    assert lib.dva_mlp_layer_bwd_supported(1000, 16, 64) == 1
    for shape in ((1000, 64, 32), (1000, 32, 128), (1000, 30, 32), (1000, 32, 33), (0, 32, 32)):
        assert lib.dva_mlp_layer_bwd_supported(*shape) == 0, shape
        assert lib.dva_mlp_layer_bwd_workspace_bytes(*shape) == 0
    assert lib.dva_mlp_layer_bwd_workspace_bytes(1000, 32, 32) >= 32 * 32 * 4
    rc = lib.dva_mlp_layer_bwd(*([None] * 11), 1000, 64, 32, 0.2, None, 0, None)
    assert rc == _lib.DVA_EUNSUPPORTED
    rc = lib.dva_mlp_layer_bwd(*([None] * 11), 1000, 32, 32, 0.2, None, 0, None)
    assert rc == _lib.DVA_EINVAL and b"mlp_layer_bwd" in lib.dva_last_error()
    # GEMM with the BatchNorm statistics in its epilogue: one column tile (N <= 128), TMA rows (multiples of 4)
    assert lib.dva_linear_bnstats_supported(1000, 128, 128) == 1
    assert lib.dva_linear_bnstats_supported(1000, 256, 128) == 0
    assert lib.dva_linear_bnstats_supported(1000, 128, 130) == 0
    assert lib.dva_linear_bnstats_workspace_bytes(128, 128) > 148 * 3 * 128 * 4


def test_no_cpu_fallback():
    import torch
    from deepviewagg_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.segment_csr(torch.zeros(3, 2), torch.tensor([0, 1, 3]), reduce="sum")
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.view_attention(torch.zeros(3, 4), torch.zeros(3, 2), torch.tensor([0, 1, 3]), 2)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "deepviewagg_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
