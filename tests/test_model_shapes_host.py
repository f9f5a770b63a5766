"""The kernel choice and workspace sizes of every model shape in model_shapes.py, without a GPU: pins the documented
envelope of the tensor-core read kernels (pmt_tc_supported) and of the tensor-core haplotype CNN (pmt_build_cnn_tc_plan),
so a change to either shows up here on every machine."""
import ctypes

import pytest
import torch

from model_shapes import ALL_SHAPES, BY_NAME, Shape, build_model
from permutect_b200.engine import library as L

CPU = torch.device("cpu")


@pytest.fixture(autouse=True)
def _restore_precision():
    yield
    L.set_precision("fp32")


def _batch(n_variants=1000, reads_per_variant=25):
    pb = L.PmtBatch()
    pb.n_variants, pb.n_rows = n_variants, n_variants * reads_per_variant
    pb.total_ref, pb.max_rows_per_variant = n_variants * 10, 40
    return pb


@pytest.mark.parametrize("shape", ALL_SHAPES, ids=lambda s: s.name)
def test_backward_kernels_in_every_precision_mode(shape):
    desc = build_model(shape, CPU).descriptor()
    L.set_precision("fp32")
    assert L.backward_kernels(desc) == {"reads_tc": False, "cnn_tc": False}
    for mode in ("tf32x3", "tf32"):
        L.set_precision(mode)
        assert L.backward_kernels(desc) == {"reads_tc": shape.bwd_tc, "cnn_tc": shape.cnn_tc}, mode


@pytest.mark.parametrize("shape", ALL_SHAPES, ids=lambda s: s.name)
def test_saved_forward_exactly_inside_both_tensor_core_envelopes(shape):
    """The training forward keeps its operands for the backward only in tf32x3, and only where both the read path and the
    CNN run on the tensor cores."""
    desc = build_model(shape, CPU).descriptor()
    pb = _batch()
    L.set_precision("tf32x3")
    saved = L.load().pmt_train_saved_bytes(ctypes.byref(desc), ctypes.byref(pb))
    assert (saved > 0) == (shape.bwd_tc and shape.cnn_tc)
    L.set_precision("fp32")
    assert L.load().pmt_train_saved_bytes(ctypes.byref(desc), ctypes.byref(pb)) == 0


@pytest.mark.parametrize("mode", ["fp32", "tf32x3"])
@pytest.mark.parametrize("shape", ALL_SHAPES, ids=lambda s: s.name)
def test_workspace_size_is_positive(shape, mode):
    desc = build_model(shape, CPU).descriptor()
    L.set_precision(mode)
    lib = L.load()
    for batch in (None, ctypes.byref(_batch())):
        for for_backward in (0, 1):
            assert lib.pmt_workspace_size(ctypes.byref(desc), batch, for_backward) > 0, (batch, for_backward)


def test_one_feature_spatial_gating_unit_is_refused():
    """self_attention_hidden_dimension 2 (H 1): the SGU LayerNorm over one feature outputs its bias whatever the input, so
    the ref reads never reach the loss; the library refuses the model instead of returning gradients that are rounding
    noise through 1 / sqrt(eps)."""
    shape = Shape("h_1", dict(BY_NAME["min_corner"].changes, self_attention_hidden_dimension=2))
    desc = build_model(shape, CPU).descriptor()
    lib = L.load()
    assert lib.pmt_workspace_size(ctypes.byref(desc), ctypes.byref(_batch()), 0) == 0
    assert b"self_attention_hidden_dimension" in lib.pmt_last_error()
    with pytest.raises(RuntimeError, match="at least 4"):
        L.backward_kernels(desc)

