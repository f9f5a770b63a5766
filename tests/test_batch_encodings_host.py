"""Batch encodings without a GPU: the kernel choice and workspace sizes for every compressed read width the header accepts
(7..15 bytes, F = 56..64), the sizes planned for a batch without a row count, and the check of a batch's read width
against the model."""
import ctypes

import numpy as np
import pytest
import torch

from model_shapes import Shape, build_model
from permutect_b200.data.batch import Batch
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.synthetic import make_arrays

CPU = torch.device("cpu")
WIDTHS = range(56, 65)


@pytest.fixture(autouse=True)
def _restore_precision():
    yield
    L.set_precision("fp32")


def _batch(n_variants, rows_per_variant, n_rows=None):
    pb = L.PmtBatch()
    pb.n_variants = n_variants
    pb.n_rows = n_variants * rows_per_variant if n_rows is None else n_rows
    pb.total_ref, pb.max_rows_per_variant = -1, rows_per_variant
    return pb


@pytest.mark.parametrize("n_read_features", WIDTHS)
def test_read_widths_kernels_and_sizes(n_read_features):
    """The tensor-core read kernels take F <= 61 (pmt_tc_supported); the CNN stays on the tensor cores at every width."""
    desc = build_model(Shape(f"f{n_read_features}", n_read_features=n_read_features), CPU).descriptor()
    assert (desc.n_read_features, desc.read_row_bytes) == (n_read_features, n_read_features - 49)
    tc = n_read_features <= 61
    lib = L.load()
    pb = _batch(1000, 25)
    for mode in ("fp32", "tf32x3", "tf32"):
        L.set_precision(mode)
        assert L.backward_kernels(desc) == {"reads_tc": tc and mode != "fp32", "cnn_tc": mode != "fp32"}, mode
        saved = lib.pmt_train_saved_bytes(ctypes.byref(desc), ctypes.byref(pb))
        assert (saved > 0) == (tc and mode == "tf32x3"), (mode, saved)
        for batch in (None, ctypes.byref(pb)):
            for for_backward in (0, 1):
                assert lib.pmt_workspace_size(ctypes.byref(desc), batch, for_backward) > 0, (mode, batch, for_backward)


@pytest.mark.parametrize("n_variants", [300, 2000, 20000])
def test_sizes_without_a_row_count_cover_sets_of_60_reads(n_variants):
    """n_rows <= 0 means "unknown": the saved training forward and the tensor-core backward's operand scratch are sized
    from a bound of the tile count, which must then hold for any rows per variant -- here sets of 60 reads, two to a
    tile, where 16 rows per variant would plan for half the tiles."""
    desc = build_model(Shape("v040"), CPU).descriptor()
    lib = L.load()
    L.set_precision("tf32x3")
    exact = _batch(n_variants, 60)
    exact_saved = lib.pmt_train_saved_bytes(ctypes.byref(desc), ctypes.byref(exact))
    exact_ws = lib.pmt_workspace_size(ctypes.byref(desc), ctypes.byref(exact), 1)
    assert exact_saved > 0 and exact_ws > 0
    for n_rows in (0, -1):
        unknown = _batch(n_variants, 60, n_rows=n_rows)
        assert lib.pmt_train_saved_bytes(ctypes.byref(desc), ctypes.byref(unknown)) >= exact_saved, n_rows
        assert lib.pmt_workspace_size(ctypes.byref(desc), ctypes.byref(unknown), 1) >= exact_ws, n_rows


def _cpu_batch(reads, n_variants=6):
    rng = np.random.default_rng(1)
    counts = np.full(n_variants, 2, np.int64)
    ia, fa, _ = make_arrays(counts, counts, rng)
    return Batch.from_arrays(ia, fa, reads[:4 * n_variants])


@pytest.mark.parametrize("reads", ["u8_11", "u8_13", "f32_60", "f16_62", "u8_1d"])
def test_batch_of_another_read_width_is_refused(reads):
    """A batch whose rows do not have the model's width (read_row_bytes compressed, n_read_features decoded) is refused
    before any library call: the kernels would read it at the model's stride."""
    model = build_model(Shape("v040"), CPU)
    desc = model.descriptor()
    kind, width = reads.split("_")
    if kind == "u8":
        rows = np.zeros((24, 12) if width == "1d" else (24, int(width)), np.uint8)
    else:
        rows = np.zeros((24, int(width)), np.float32 if kind == "f32" else np.float16)
    batch = _cpu_batch(rows)
    if width == "1d":
        batch.reads = batch.reads.reshape(-1)
    flat = model.flat_weights().detach()
    zeros = torch.zeros((batch.size(), desc.n_clusters + 2))
    with pytest.raises(ValueError, match="do not match the model"):
        engine.forward_call(desc, flat, batch)
    with pytest.raises(ValueError, match="do not match the model"):
        engine.backward_call(desc, flat, batch, zeros, None, None)
    with pytest.raises(ValueError, match="do not match the model"):
        engine.head_backward_call(desc, flat, batch, torch.zeros((24, desc.d_feat)), zeros, None, None)


@pytest.mark.parametrize("reads", [np.zeros((24, 12), np.uint8), np.zeros((24, 61), np.float32), np.zeros((24, 61), np.float16)],
                         ids=["u8_12", "f32_61", "f16_61"])
def test_batch_of_the_model_read_width_passes_the_check(reads):
    """Rows of the model's width get past the check (and then to the CUDA-only refusal of a CPU call)."""
    model = build_model(Shape("v040"), CPU)
    with pytest.raises(RuntimeError, match="CUDA devices only"):
        engine.forward_call(model.descriptor(), model.flat_weights().detach(), _cpu_batch(reads))
