"""FlatAdamW (pmt_adamw_step through the C-ABI) against torch's clip_grad_norm_ + AdamW on the same gradients,
including frozen parameters (calibration epochs) and several steps of moment state."""
import numpy as np
import pytest
import torch

from golden_utils import load
from helpers import golden_batch, model_from_golden
from permutect_b200.training.step import FlatAdamW, backpropagate, make_optimizer
from permutect_b200.utils.enums import Epoch

pytestmark = pytest.mark.gpu


def _models():
    g = load("v040_seed0_b64")
    dev = torch.device("cuda:0")
    a, b = model_from_golden(g, dev), model_from_golden(g, dev)
    return g, a, b


def test_flat_adamw_matches_torch_clip_and_adamw():
    g, ma, mb = _models()
    opt_a = make_optimizer(ma, learning_rate=3e-3, weight_decay=0.02)
    assert isinstance(opt_a, FlatAdamW)
    opt_b = torch.optim.AdamW(mb.parameters(), lr=3e-3, weight_decay=0.02)
    gen = torch.Generator().manual_seed(0)
    for step in range(4):
        scale = [30.0, 0.01, 1.0, 5.0][step]        # exercise both sides of the clip threshold
        for (na, pa), (nb, pb) in zip(ma.named_parameters(), mb.named_parameters()):
            gr = (torch.randn(pa.shape, generator=gen) * scale).to(pa.device)
            pa.grad, pb.grad = gr.clone(), gr.clone()
        if step == 2:                                # a frozen tensor: no gradient on either side
            ma.feature_clustering.artifact_emg.mu_k.grad = None
            mb.feature_clustering.artifact_emg.mu_k.grad = None
        norm_b = torch.nn.utils.clip_grad_norm_(list(mb.parameters()), max_norm=1.0)
        opt_b.step()
        opt_a.step()
        assert abs(float(opt_a.total_norm) - float(norm_b)) <= 1e-5 * float(norm_b)
        for (na, pa), (nb, pb) in zip(ma.named_parameters(), mb.named_parameters()):
            torch.testing.assert_close(pa, pb, rtol=2e-6, atol=2e-7, msg=lambda m: f"step {step} {na}: {m}")


def test_training_step_with_flat_optimizer_changes_the_forward():
    g, model, _ = _models()
    dev = model._device
    model.set_epoch_type(Epoch.TRAIN)
    opt = make_optimizer(model)
    batch = golden_batch(g, dev)
    losses0 = model.compute_batch_losses(model.compute_batch_output(batch), batch)
    first = float(losses0.total_loss.detach())
    backpropagate(opt, losses0.total_loss, params_to_clip=model.parameters())
    for _ in range(5):
        losses = model.compute_batch_losses(model.compute_batch_output(batch), batch)
        backpropagate(opt, losses.total_loss, params_to_clip=model.parameters())
    model.set_epoch_type(Epoch.VALID)
    with torch.inference_mode():                    # the cached materialised weights must see the in-place updates
        out = model.compute_batch_output(batch)
        last = float(model.compute_batch_losses(out, batch).total_loss)
    assert np.isfinite(last) and last < first
    sd = model.state_dict()                         # parameters are views of the flat buffer: state dict unchanged in form
    assert set(sd.keys()) == set(g.sd.keys())


def test_flat_gradient_path_equals_per_parameter_path():
    """make_optimizer attaches the model to the optimiser's flat buffers (one gradient tensor instead of ~190
    accumulations); the weights it produces must be those of the per-parameter autograd path, also when only the
    calibration parameters train (model_training.py:137-139) and when two backward passes accumulate."""
    from permutect_b200.utils.enums import Epoch as E
    g, ma, mb = _models()
    dev = ma._device
    batch = golden_batch(g, dev)
    opts = []
    for m, attached in ((ma, True), (mb, False)):
        m.set_epoch_type(E.TRAIN)
        opt = make_optimizer(m, learning_rate=2e-3, weight_decay=0.01)
        assert m._flat_optimizer is opt
        if not attached:
            m._flat_optimizer = None
        opts.append(opt)

    def step(m, opt, accumulate=False):
        opt.zero_grad(set_to_none=True)
        for _ in range(2 if accumulate else 1):
            m.compute_batch_losses(m.compute_batch_output(batch), batch).total_loss.backward()
        opt.step()

    def compare(tag):
        for (na, pa), (nb, pb) in zip(ma.named_parameters(), mb.named_parameters()):
            # the flat path evaluates the constraint maps in pmt_constraints_forward (warp-tree sums), the per-parameter path
            # in torch: norms and log-sum-exps differ in the last place, which Adam's g / sqrt(v) carries into the weights
            torch.testing.assert_close(pa, pb, rtol=5e-6, atol=5e-7, msg=lambda msg: f"{tag} {na}: {msg}")

    for i in range(3):
        step(ma, opts[0]); step(mb, opts[1])
        compare(f"step {i}")
    assert ma.read_embedding._model[0].weight.grad.data_ptr() != mb.read_embedding._model[0].weight.grad.data_ptr()
    assert opts[0]._flat_grad_valid and not opts[1]._flat_grad_valid
    step(ma, opts[0], accumulate=True); step(mb, opts[1], accumulate=True)
    compare("accumulated")
    for m in (ma, mb):                                   # calibration epoch
        for p in m.parameters():
            p.requires_grad = False
        for p in m.calibration_parameters():
            p.requires_grad = True
    frozen_before = ma.read_embedding._model[0].weight.detach().clone()
    for i in range(2):
        step(ma, opts[0]); step(mb, opts[1])
        compare(f"calibration step {i}")
    assert torch.equal(frozen_before, ma.read_embedding._model[0].weight.detach())


def test_rotation_kernels_match_the_torch_formulation():
    """pmt_orthogonal_forward / _backward against the float64 scaling-and-squaring written with torch ops (itself checked
    against the reference's orthogonal parametrisation by the golden fixtures), with and without a base matrix."""
    from permutect_b200.engine import plan as planner
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(4)
    for n in (1, 3, 10, 16):
        for with_base in (False, True):
            X = (torch.randn((n, n), generator=gen) * 1.5).to(dev).requires_grad_(True)
            base = None
            if with_base:
                base = torch.linalg.qr(torch.randn((n, n), generator=gen))[0].to(dev)
            Q = planner._RotationFunction.apply(X, base)
            Xl = X.detach().double().tril().requires_grad_(True)
            A = Xl - Xl.mT
            want = torch.matrix_exp(A)
            if with_base:
                want = base.double() @ want
            torch.testing.assert_close(Q.double(), want.detach(), rtol=1e-5, atol=2e-6)
            torch.testing.assert_close((Q @ Q.mT).cpu(), torch.eye(n), rtol=0, atol=1e-5)
            dQ = torch.randn((n, n), generator=gen).to(dev)
            Q.backward(dQ)
            want.backward(dQ.double())
            torch.testing.assert_close(X.grad.double(), Xl.grad.tril(), rtol=1e-4, atol=1e-5)


def _check_flat_materialisation(model):
    """engine/plan.py:_FastMaterialize (pmt_constraints_forward / _backward and the rotation) against torch.cat of the
    parametrised tensors (utils/parameterizations.py) and autograd through them; the rotation's slot of the gradient bit
    for bit, since it is the same calls on the same dQ as autograd through _orthogonal_without_sync."""
    from permutect_b200.engine import plan as planner

    params = list(model.parameters())
    opt = FlatAdamW(params)
    opt.attach(model)
    received = {}
    opt.receive_flat_gradient = lambda g: received.__setitem__("g", g)

    w_fast = planner.materialize_flat(opt)
    w_ref = torch.cat([t.reshape(-1) for t in planner.materialized_tensors(model)])
    torch.testing.assert_close(w_fast, w_ref, rtol=2e-6, atol=1e-7)
    dw = torch.randn_like(w_ref)
    w_ref.backward(dw)
    want = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
    for p in params:
        p.grad = None
    w_fast.backward(dw)
    got = received["g"]
    torch.testing.assert_close(got, want, rtol=1e-5, atol=1e-6)
    _, _, _, off, n = opt._constraint_pack.rotation
    assert torch.equal(got[off:off + n], want[off:off + n])


def test_flat_materialisation_matches_the_autograd_formulation():
    """The v0.4.0 model: the rotation (10 x 10) through pmt_orthogonal_forward / _backward."""
    import bench
    torch.manual_seed(0)
    model = bench.make_model(torch.device("cuda:0"))
    with torch.no_grad():
        for p in model.parameters():
            p.add_(0.1 * torch.randn_like(p))
    _check_flat_materialisation(model)


def test_flat_materialisation_with_the_float64_rotation_matches_the_autograd_formulation():
    """d_feat 17 (model_shapes.py's e_17): the rotation is past the kernel pair's n <= 16 and takes the float64
    scaling-and-squaring inside the node."""
    from model_shapes import BY_NAME, build_model
    _check_flat_materialisation(build_model(BY_NAME["e_17"], torch.device("cuda:0")))
