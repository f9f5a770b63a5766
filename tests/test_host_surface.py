"""CPU-only checks of the drop-in surface: state-dict compatibility with the reference, the kernel
descriptor, the .pt format, and that the C-ABI library loads and exports what the header declares."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from golden_utils import CASES, load
from helpers import model_from_golden, params_from_hp
from permutect_b200.architecture.artifact_model import ArtifactModel, load_model
from permutect_b200.engine import library as L
from permutect_b200.engine import plan as planner

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPU = torch.device("cpu")


@pytest.mark.parametrize("case", CASES)
def test_state_dict_keys_and_shapes_match_reference(case):
    g = load(case)
    model = model_from_golden(g, CPU)      # load_state_dict(strict=True) inside
    sd = model.state_dict()
    assert list(sd.keys()) == list(g.sd.keys())
    for k, v in g.sd.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    names = [n for n, _ in model.named_parameters()]
    assert names == list(g.grad.keys())     # same order as the reference's named_parameters()


def test_same_seed_gives_reference_initial_weights():
    g = load("v040_seed0_b64")
    torch.manual_seed(0)
    model = ArtifactModel(params_from_hp(g.hp), 61, 71, 42, device=CPU)
    for k, v in model.state_dict().items():
        torch.testing.assert_close(v, g.sd[k], rtol=0, atol=0, msg=k)


def test_parameter_count_v040():
    g = load("v040_seed0_b64")
    model = model_from_golden(g, CPU)
    assert sum(p.numel() for p in model.parameters()) == 68229       # SURVEY.md Appendix B
    assert len(list(model.parameters())) == 194
    assert sum(v.numel() for v in model.state_dict().values()) == 68329


def test_descriptor_v040():
    g = load("v040_seed0_b64")
    model = model_from_golden(g, CPU)
    d = planner.build_desc(model)
    assert (d.n_read_features, d.read_row_bytes, d.n_info_features, d.hap_len) == (61, 12, 71, 21)
    assert (d.d_read, d.d_info, d.d_seq, d.d_model, d.d_ffn, d.n_blocks, d.d_feat, d.n_clusters) == (30, 20, 10, 60, 20, 6, 10, 4)
    assert d.n_params == 68229
    assert (d.n_read_ops, d.n_info_ops, d.n_red_ops) == (7, 7, 5)
    ops = [d.read_ops[i] for i in range(d.n_read_ops)]
    assert (ops[0].in_dim, ops[0].out_dim, ops[0].w_off, ops[0].b_off, ops[0].flags) == (61, 30, 0, 1830, L.OP_POST_SELU)
    assert ops[1].flags == L.OP_SKIP_BEGIN | L.OP_POST_SELU and ops[2].flags == L.OP_SKIP_END
    assert ops[1].alpha_off == 1860 and ops[1].w_off == 1861          # Appendix B offsets
    red = [d.red_ops[i] for i in range(d.n_red_ops)]
    assert red[0].alpha_off == 49632 and red[4].w_off == 64274 and red[4].flags == 0
    assert d.blocks[0].ln_w == 26136 and d.blocks[0].reg_weight == 26136 + 2595
    assert d.translation == 64884 and d.rotation == 64894 and d.sigma_e == 64994 and d.unit_ke == 65004
    cnn = [d.cnn_ops[i] for i in range(d.n_cnn_ops)]
    assert [c.kind for c in cnn] == [1, 2, 1, 2, 1, 2, 1, 2, 3]
    assert [c.act for c in cnn if c.kind == 1] == [L.ACT_SELU] * 4
    assert [(c.in_len, c.out_len) for c in cnn[:8]] == [(21, 19), (19, 18), (18, 16), (16, 16), (16, 12), (12, 6), (6, 2), (2, 1)]


def test_descriptor_small_hp_folds_activation_over_pool():
    g = load("small_hp")
    d = planner.build_desc(model_from_golden(g, CPU))
    cnn = [d.cnn_ops[i] for i in range(d.n_cnn_ops)]
    assert [c.kind for c in cnn] == [1, 2, 3]
    assert cnn[0].act == L.ACT_LEAKY_RELU and cnn[0].out_ch == 64 and cnn[1].out_len == 9 and cnn[2].in_ch == 576
    assert all(d.read_ops[i].flags == (L.OP_POST_SELU if i < 2 else 0) for i in range(3))


def test_materialised_weights_follow_the_constraints():
    g = load("v040_perturbed_edge")
    model = model_from_golden(g, CPU)
    d = planner.build_desc(model)
    flat = torch.cat([t.reshape(-1) for t in planner.materialized_tensors(model)]).detach()
    assert flat.numel() == d.n_params
    sigma = flat[d.sigma_e:d.sigma_e + 10]
    raw = g.sd["feature_clustering.parametrizations.nonartifact_stdev_e.original"]
    torch.testing.assert_close(sigma, 99.99 * torch.sigmoid(raw) + 0.01)
    unit = flat[d.unit_ke:d.unit_ke + 40].view(4, 10)
    torch.testing.assert_close(unit.norm(dim=-1), torch.ones(4))
    q = flat[d.rotation:d.rotation + 100].view(10, 10)
    torch.testing.assert_close(q @ q.t(), torch.eye(10), atol=1e-5, rtol=0)
    torch.testing.assert_close(flat[d.logw_k:d.logw_k + 4].exp().sum(), torch.tensor(1.0))
    rw = g.sd["ref_alt_reads_encoder.blocks.2.sgu.parametrizations.reg_weight.original"]
    torch.testing.assert_close(flat[d.blocks[2].reg_weight], torch.exp(rw))


def test_save_load_roundtrip_and_pickle_path(tmp_path):
    g = load("v040_two_sources")
    model = model_from_golden(g, CPU)
    path = tmp_path / "model.pt"
    model.save_model(path)                      # resets the source predictor to one source (artifact_model.py:341)
    raw = open(path, "rb").read()
    import sys
    if getattr(sys.modules.get("permutect.parameters"), "_permutect_b200_alias", False):
        assert b"permutect.parameters" in raw or b"permutect\nparameters" in raw or re.search(rb"permutect.{0,4}parameters", raw)
    else:     # an earlier test imported the real reference (oracle/reference.py:load): the alias is retired in this process
        assert re.search(rb"permutect_b200.{0,4}parameters", raw)
    loaded, priors, spectra = load_model(path, device=CPU)
    assert priors is None and spectra is None and loaded.num_sources == 1
    for k, v in loaded.state_dict().items():
        torch.testing.assert_close(v, model.state_dict()[k], rtol=0, atol=0)
    assert loaded._params.read_layers == g.hp["read_layers"]


def test_calibration_parameters_and_epoch_freezing():
    from permutect_b200.utils.enums import Epoch
    model = model_from_golden(load("v040_seed0_b64"), CPU)
    cal = model.calibration_parameters()
    assert [tuple(p.shape) for p in cal] == [(10,), (4,)]
    model.set_epoch_type(Epoch.VALID)
    assert not any(p.requires_grad for p in model.parameters()) and not model.training
    model.set_epoch_type(Epoch.TRAIN)
    assert all(p.requires_grad for p in model.parameters()) and model.training


def test_unsupported_options_fail_loudly():
    hp = dict(load("small_hp").hp)
    hp["batch_normalize"] = True
    with pytest.raises(NotImplementedError):
        ArtifactModel(params_from_hp(hp), 61, 71, 42, device=CPU)


def test_layers_have_no_eager_forward():
    model = model_from_golden(load("small_hp"), CPU)
    with pytest.raises(RuntimeError):
        model.read_embedding(torch.zeros(2, 61))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(REPO, "include", "permutect_b200.h")).read()
    declared = set(re.findall(r"\b(pmt_[a-z_]+)\s*\(", header))
    assert declared == set(L.EXPORTED_SYMBOLS)
    lib = L.load()
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.pmt_abi_version() == L.PMT_ABI_VERSION


def test_ctypes_structs_match_header_sizes():
    # sizes computed from the header's field lists (all int32 unless noted)
    assert ctypes.sizeof(L.PmtLinearOp) == 24 and ctypes.sizeof(L.PmtCnnOp) == 40 and ctypes.sizeof(L.PmtBlockOffsets) == 76
    assert ctypes.sizeof(L.PmtModelDesc) == 17 * 4 + 3 * 16 * 24 + 16 * 40 + 12 * 76 + 10 * 4
    assert ctypes.sizeof(L.PmtBatch) == 16 + 3 * 8 + 4 * 8 + 8 + 8 + 8 + 8
    assert ctypes.sizeof(L.PmtOutputs) == 7 * 8 and ctypes.sizeof(L.PmtOutGrads) == 5 * 8


def test_ctypes_structs_match_the_compiled_header(tmp_path):
    """sizeof of every structure of include/permutect_b200.h as gcc lays it out == the ctypes mirror."""
    import os
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    names = ["PmtLinearOp", "PmtCnnOp", "PmtBlockOffsets", "PmtModelDesc", "PmtBatch", "PmtOutputs", "PmtOutGrads",
             "PmtLossDesc", "PmtLossBatch", "PmtLossOutputs", "PmtLossGrads", "PmtPosteriorDesc", "PmtPosteriorOutputs",
             "PmtConstraintGroup"]
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "sizes.c"
    src.write_text('#include <stdio.h>\n#include "permutect_b200.h"\nint main(void) {\n' +
                   "".join(f'  printf("{n} %zu\\n", sizeof({n}));\n' for n in names) + "  return 0;\n}\n")
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", "-I", os.path.join(repo, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    got = dict(line.split() for line in out.strip().splitlines())
    for n in names:
        assert int(got[n]) == ctypes.sizeof(getattr(L, n)), n


def test_workspace_size_is_positive_without_a_gpu():
    model = model_from_golden(load("v040_seed0_b64"), CPU)
    d = planner.build_desc(model)
    pb = L.PmtBatch()
    pb.n_variants = 1000
    assert L.load().pmt_workspace_size(ctypes.byref(d), ctypes.byref(pb), 0) > 0


def test_compute_requires_cuda():
    from helpers import golden_batch
    g = load("v040_seed0_b64")
    model = model_from_golden(g, CPU)
    with pytest.raises(RuntimeError):
        model.compute_batch_output(golden_batch(g, None))


def test_sync_free_rotation_equals_torch_orthogonal():
    """engine/plan.py evaluates the orthogonal parametrisation without torch.matrix_exp (which synchronises the device);
    value and gradient must agree with torch's own."""
    from permutect_b200.engine.plan import _orthogonal_without_sync
    model = model_from_golden(load("v040_seed0_b64"), CPU)
    rot = model.pre_clustering_transform.rotation_ee
    gen = torch.Generator().manual_seed(0)
    for scale in (0.0, 0.3, 2.0, 6.0):
        with torch.no_grad():
            rot.parametrizations.weight.original.copy_(scale * torch.randn(rot.parametrizations.weight.original.shape, generator=gen))
        want = rot.weight
        got = _orthogonal_without_sync(rot, "weight")
        assert got is not None
        torch.testing.assert_close(got, want, rtol=0, atol=3e-6)
        torch.testing.assert_close(got @ got.T, torch.eye(got.shape[0]), rtol=0, atol=5e-6)
        w = torch.randn(want.shape, generator=gen)
        g_want, = torch.autograd.grad((want * w).sum(), rot.parametrizations.weight.original)
        g_got, = torch.autograd.grad((got * w).sum(), rot.parametrizations.weight.original)
        torch.testing.assert_close(g_got, g_want, rtol=1e-4, atol=1e-5)

