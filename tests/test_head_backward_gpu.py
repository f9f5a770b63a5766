"""Calibration epochs and head-only training: pmt_head_backward instead of the whole model's backward.

When no tensor upstream of the rotation trains (read_embedding, info_embedding, haplotypes_cnn, ref_alt_reads_encoder,
reducer), compute_batch_output keeps the forward's per-read final features and its backward is pmt_head_backward: no
saved training forward, no pmt_backward.  The gradients are checked against the float64 oracle at the model shapes of
model_shapes.py, including the shapes whose full backward refuses (trains=False), against the full path, on sets longer
than a tile and downsampled batches, run to run, through run_epoch and through a CUDA-graph replay."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from helpers import batch_from_raw
from model_shapes import BY_NAME, Shape, long_set_raw, make_raw
from oracle import artifact_oracle as orc
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.utils.enums import Epoch
from test_model_shapes_gpu import DEV, LONG_SHAPES, SIZES, Case, _report

pytestmark = pytest.mark.gpu
TRUNK = ("read_embedding", "info_embedding", "haplotypes_cnn", "ref_alt_reads_encoder", "reducer")
V040 = Shape("v040")
CALIBRATION_SHAPES = [V040, BY_NAME["min_corner"], BY_NAME["deep_odd"], BY_NAME["e1"], BY_NAME["max_corner"], BY_NAME["h_12"],
                      BY_NAME["simt_limits"]]
CONTRACT = {"fp32": 2e-3, "tf32x3": 4e-3}


@pytest.fixture(autouse=True)
def _restore():
    yield
    L.set_precision("fp32")


@pytest.fixture
def calls(monkeypatch):
    """Counts pmt_backward calls and training forwards that ask for the saved forward."""
    seen = {"backward": 0, "saved_forward": 0}
    backward_call, forward_call = engine.backward_call, engine.forward_call

    def spy_backward(*a, **k):
        seen["backward"] += 1
        return backward_call(*a, **k)

    def spy_forward(*a, **k):
        seen["saved_forward"] += bool(k.get("for_training"))
        return forward_call(*a, **k)

    monkeypatch.setattr(engine, "backward_call", spy_backward)
    monkeypatch.setattr(engine, "forward_call", spy_forward)
    return seen


def calibration_names(model):
    ids = {id(p) for p in model.calibration_parameters()}
    return {n for n, p in model.named_parameters() if id(p) in ids}


def head_names(model):
    """Every tensor downstream of the trunk: translation, rotation, the clustering head and the adversarial heads."""
    return {n for n, _ in model.named_parameters() if not n.startswith(TRUNK)}


def gradients(model, batch, mode, trainable):
    """One training step's backward with exactly `trainable` requiring grad: {name: grad or None}."""
    L.set_precision(mode)
    model.set_epoch_type(Epoch.TRAIN)
    for n, p in model.named_parameters():
        p.requires_grad = n in trainable
        p.grad = None
    out = model.compute_batch_output(batch)
    model.compute_batch_losses(out, batch).total_loss.backward()
    torch.cuda.synchronize()
    return {n: (None if p.grad is None else p.grad.detach().cpu().numpy().copy()) for n, p in model.named_parameters()}


def check_against_oracle(case, got, trainable, mode, what):
    """Each trainable tensor within the contract of its largest entry; the frozen ones have no gradient."""
    assert all(got[n] is None for n in got if n not in trainable)
    rel = {n: float(np.abs(got[n] - case.want_grads[n]).max()) / max(float(np.abs(case.want_grads[n]).max()), 1e-3)
           for n in trainable}
    _report(case, f"{mode} {what}", {"worst relative-to-max": max(rel.values())})
    bad = sorted(((e, n) for n, e in rel.items() if e > CONTRACT[mode]), reverse=True)
    assert not bad, f"{mode} {what} gradient error too large:\n" + "\n".join(f"{e:.3e} {n}" for e, n in bad)


def _calibration_params():
    for shape in CALIBRATION_SHAPES:
        for n in SIZES:
            for mode in ("fp32", "tf32x3") if shape.reads_tc else ("fp32",):
                yield pytest.param(shape, n, mode, id=f"{shape.name}-{n}-{mode}")


@pytest.mark.parametrize("shape,n_variants,mode", list(_calibration_params()))
def test_calibration_gradients_against_float64(shape, n_variants, mode, calls):
    """Only calibration_parameters() train: at every shape, the ones whose full backward refuses included."""
    case = Case(shape, make_raw(shape, n_variants, seed=50 + n_variants), grads=True, key=("head", n_variants))
    trainable = calibration_names(case.model)
    assert len(trainable) == 2
    got = gradients(case.model, case.batch, mode, trainable)
    check_against_oracle(case, got, trainable, mode, "calibration")
    assert calls == {"backward": 0, "saved_forward": 0}


@pytest.mark.parametrize("shape", [V040, BY_NAME["deep_odd"]], ids=lambda s: s.name)
@pytest.mark.parametrize("mode", ["fp32", "tf32x3"])
def test_every_head_tensor_against_float64(shape, mode, calls):
    """Translation, rotation, every clustering parameter and both adversarial heads train with the trunk frozen: dt and dQ
    also carry the gradient of the alt means that the adversarial heads send back."""
    case = Case(shape, make_raw(shape, 5000, seed=60), grads=True, key=("head", "all"))
    trainable = head_names(case.model)
    got = gradients(case.model, case.batch, mode, trainable)
    assert case.model.trunk_frozen()
    check_against_oracle(case, got, trainable, mode, "head tensors")
    assert any(n.startswith("pre_clustering_transform") for n in trainable)
    assert calls == {"backward": 0, "saved_forward": 0}


@pytest.mark.parametrize("shape", [V040, BY_NAME["deep_odd"]], ids=lambda s: s.name)
def test_head_path_agrees_with_the_full_backward(shape, calls):
    """Unfreezing the reducer's last bias sends the same step through pmt_backward; the head tensors' gradients of both
    paths agree to 1e-5 of each tensor's largest entry (fp32)."""
    raw = make_raw(shape, 5000, seed=70)
    case = Case(shape, raw)
    heads = head_names(case.model)
    last_bias = [n for n, _ in case.model.named_parameters() if n.startswith("reducer") and n.endswith("bias")][-1]
    head = gradients(case.model, case.batch, "fp32", heads)
    assert calls["backward"] == 0
    full = gradients(case.model, case.batch, "fp32", heads | {last_bias})
    assert calls["backward"] == 1
    rel = {n: float(np.abs(head[n] - full[n]).max()) / max(float(np.abs(full[n]).max()), 1e-30) for n in heads}
    _report(case, "head path vs pmt_backward", {"worst relative-to-max": max(rel.values())})
    bad = sorted(((e, n) for n, e in rel.items() if e > 1e-5), reverse=True)
    assert not bad, "\n".join(f"{e:.3e} {n}" for e, n in bad)


@pytest.mark.parametrize("shape", [V040, BY_NAME["max_corner"]], ids=lambda s: s.name)
def test_long_sets_against_float64(shape, calls):
    """Sets of up to 4 400 reads, sets without ref reads, tf32x3: the final features come from the tensor-core long-set
    forward."""
    case = Case(shape, long_set_raw(shape, LONG_SHAPES, seed=13), grads=True, key=("head", "long"))
    trainable = head_names(case.model)
    got = gradients(case.model, case.batch, "tf32x3", trainable)
    check_against_oracle(case, got, trainable, "tf32x3", "long sets")
    assert calls == {"backward": 0, "saved_forward": 0}


@pytest.mark.parametrize("mode", ["fp32", "tf32x3"])
def test_downsampled_batch_against_float64(mode):
    """A DownsampledBatch: rows reach the kernels through read_indices (quirk Q1); the oracle gathers the same rows."""
    from model_shapes import build_model
    from permutect_b200.data.batch import DownsampledBatch
    raw = make_raw(V040, 2000, seed=80)
    frac = torch.full((2000,), 0.6, device=DEV)
    ds = DownsampledBatch(batch_from_raw(raw, DEV), frac, frac, seed=5)
    ref_c, alt_c = ds.counts()
    n = int(ref_c.sum() + alt_c.sum())
    ds_raw = dict(raw, read_indices=ds.read_indices[:n].cpu().numpy(), ref_counts=ref_c.cpu().numpy().astype(np.int64),
                  alt_counts=alt_c.cpu().numpy().astype(np.int64))
    model = build_model(V040, DEV)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    names = [k for k, _ in model.named_parameters()]
    _, _, want = orc.loss_and_grads(sd, V040.hp, ds_raw, names, dtype=torch.float64, num_sources=1,
                                    source_adversarial_strength=0.3)
    case = SimpleNamespace(shape=V040, raw=ds_raw, want_grads={k: v.numpy() for k, v in want.items()})
    trainable = head_names(model)
    got = gradients(model, ds, mode, trainable)
    check_against_oracle(case, got, trainable, mode, "downsampled")


def test_bitwise_reproducible(calls):
    case = Case(V040, make_raw(V040, 5000, seed=90))
    trainable = head_names(case.model)
    a = gradients(case.model, case.batch, "tf32x3", trainable)
    b = gradients(case.model, case.batch, "tf32x3", trainable)
    for n in trainable:
        np.testing.assert_array_equal(a[n], b[n], err_msg=n)
    assert calls == {"backward": 0, "saved_forward": 0}


class _Downsampler:
    def calculate_downsampling_fractions(self, batch):
        f = torch.full((batch.size(),), 0.7)
        return f, f


def test_calibration_epoch_moves_only_the_calibration_tensors(calls):
    """run_epoch(is_calibration_epoch=True) with FlatAdamW: every step goes through the head path and only the two
    calibration tensors change."""
    import bench
    from permutect_b200.data.batch import Batch
    from permutect_b200.synthetic import make_wgs_arrays
    from permutect_b200.training import model_training as mt
    from permutect_b200.training.step import make_optimizer
    torch.manual_seed(0)
    model = bench.make_model(DEV)
    L.set_precision("tf32x3")
    opt = make_optimizer(model)
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    loader = [Batch.from_arrays(*make_wgs_arrays(300, seed=s)) for s in (1, 2)]
    assert mt.run_epoch(model, loader, _Downsampler(), Epoch.TRAIN, optimizer=opt, is_calibration_epoch=True) == 4
    calibration = calibration_names(model)
    for n, p in model.named_parameters():
        moved = not torch.equal(p.detach(), before[n])
        assert moved == (n in calibration), n
    assert calls == {"backward": 0, "saved_forward": 0}


@pytest.mark.parametrize("shape", [V040, BY_NAME["max_corner"]], ids=lambda s: s.name)
def test_graphed_calibration_step_equals_eager_step(shape):
    """GraphedTrainStep captures the head path (at the max corner too, where a full step cannot run) and its replays give
    the eager steps' losses and weights bitwise."""
    from permutect_b200.data.batch import DownsampledBatch
    from permutect_b200.engine.graphs import GraphedTrainStep
    from permutect_b200.training.model_training import freeze, unfreeze
    from permutect_b200.training.step import make_optimizer, train_step
    from helpers import params_from_hp
    from model_shapes import build_model
    from permutect_b200.architecture.artifact_model import ArtifactModel
    L.set_precision("tf32x3")
    parent = batch_from_raw(make_raw(shape, 256, seed=95), DEV)
    frac = torch.full((256,), 0.8, device=DEV)
    example = DownsampledBatch(parent, frac, frac, seed=1)
    batches = [DownsampledBatch(parent, frac, frac, seed=100 + i) for i in range(4)]

    def run(graphed):
        model = ArtifactModel(params_from_hp(shape.hp), 61, shape.n_info, 2 * shape.hap_len, device=DEV)   # built on the GPU
        model.load_state_dict(build_model(shape, DEV).state_dict())
        model.set_epoch_type(Epoch.TRAIN)
        freeze(model.parameters())
        unfreeze(model.calibration_parameters())
        opt = make_optimizer(model, learning_rate=1e-2, weight_decay=0.01)
        step = GraphedTrainStep(model, opt, example) if graphed else None
        losses = [float(step(b)) if graphed else float(train_step(model, b, opt)[1].total_loss.detach()) for b in batches]
        return losses, opt.flat.detach().cpu().numpy().copy()

    l_eager, w_eager = run(False)
    l_graph, w_graph = run(True)
    assert l_eager == l_graph
    np.testing.assert_array_equal(w_eager, w_graph)
