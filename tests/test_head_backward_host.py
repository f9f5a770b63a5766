"""The head-only backward's host surface, without a GPU: its workspace size at every model shape the library accepts
(those whose full backward refuses included) and the trunk-frozen predicate that selects it."""
import ctypes

import pytest
import torch

from model_shapes import ALL_SHAPES, BY_NAME, build_model
from permutect_b200.engine import library as L

CPU = torch.device("cpu")
TRUNK = ("read_embedding", "info_embedding", "haplotypes_cnn", "ref_alt_reads_encoder", "reducer")


@pytest.mark.parametrize("shape", ALL_SHAPES, ids=lambda s: s.name)
def test_workspace_size_at_every_shape(shape):
    desc = build_model(shape, CPU).descriptor()
    assert L.load().pmt_head_backward_workspace_size(ctypes.byref(desc)) > 0


def test_workspace_size_refuses_a_bad_descriptor():
    desc = build_model(BY_NAME["min_corner"], CPU).descriptor()
    desc.abi_version = 2
    lib = L.load()
    assert lib.pmt_head_backward_workspace_size(ctypes.byref(desc)) == 0
    assert "abi_version" in lib.pmt_last_error().decode()


@pytest.mark.parametrize("module", TRUNK + (None,))
def test_trunk_frozen_only_when_all_five_trunk_modules_are(module):
    """Every tensor downstream of the trunk trains; `module` unfreezes one tensor of one trunk module (None: none)."""
    model = build_model(BY_NAME["min_corner"], CPU)
    for name, p in model.named_parameters():
        p.requires_grad = not name.startswith(TRUNK)
    if module is not None:
        next(getattr(model, module).parameters()).requires_grad = True
    assert model.trunk_frozen() == (module is None)
