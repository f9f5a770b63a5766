"""Pins oracle/artifact_oracle.py against the reference-generated golden fixtures (CPU only)."""
import numpy as np
import pytest
import torch

from golden_utils import CASES, load
from oracle import artifact_oracle as orc


@pytest.mark.parametrize("case", CASES)
def test_decode_matches_reference(case):
    g = load(case)
    np.testing.assert_array_equal(orc.decode_reads(g.inputs["reads_u8"]), g.inputs["decoded_reads"])


def test_decode_wraps_like_reference():
    # SURVEY.md §9 Q2: dec([0,96,127,128,160,255]) = [4.0, 7.0, 7.97, 0.0, 1.0, 3.97]
    row = np.zeros((6, 12), np.uint8)
    row[:, 7] = [0, 96, 127, 128, 160, 255]
    np.testing.assert_allclose(orc.decode_reads(row)[:, 56], [4.0, 7.0, 7.96875, 0.0, 1.0, 3.96875])


@pytest.mark.parametrize("case", CASES)
def test_forward_and_losses_match_reference(case):
    g = load(case)
    with torch.no_grad():
        out = orc.forward(g.sd, g.hp, g.raw())
        ls = orc.losses(g.sd, g.hp, g.raw(), out, num_sources=g.hp["num_sources"],
                        source_adversarial_strength=g.hp["source_adversarial_strength"])
    for k, want in g.out.items():
        np.testing.assert_allclose(out[k].numpy(), want, rtol=2e-5, atol=2e-5, err_msg=k)
    for k, want in g.loss.items():
        np.testing.assert_allclose(ls[k].numpy(), want, rtol=2e-5, atol=2e-5, err_msg=k)


def test_smoke_value_from_survey():
    g = load("v040_seed0_b64")
    with torch.no_grad():
        out = orc.forward(g.sd, g.hp, g.raw())
    np.testing.assert_allclose(out["logits_b"][:5].numpy(), [-13.2103, -4.3585, -15.9768, -15.3913, -18.4226], atol=2e-4)


@pytest.mark.parametrize("case", CASES)
def test_gradients_match_reference(case):
    g = load(case)
    trainable = list(g.grad.keys())
    _, _, grads = orc.loss_and_grads(g.sd, g.hp, g.raw(), trainable, num_sources=g.hp["num_sources"],
                                     source_adversarial_strength=g.hp["source_adversarial_strength"])
    for k, want in g.grad.items():
        got = grads[k].numpy()
        scale = max(1.0, float(np.abs(want).max()))
        np.testing.assert_allclose(got, want, rtol=1e-3, atol=2e-5 * scale, err_msg=k)


@pytest.mark.parametrize("case", CASES)
def test_float64_oracle_computes_the_same_function(case):
    """The double-precision oracle (the reference the kernel tests measure against) agrees with the float32 one, which the
    fixtures pin, to float32 rounding: forward values, losses and every parameter gradient.  The absolute 1e-4 is the
    float32 rounding accumulated over ~45 layers (measured up to 3.3e-5 on a logit), a tenth of the kernels' contract."""
    g = load(case)
    trainable = list(g.grad.keys())
    kw = dict(num_sources=g.hp["num_sources"], source_adversarial_strength=g.hp["source_adversarial_strength"])
    out32, ls32, gr32 = orc.loss_and_grads(g.sd, g.hp, g.raw(), trainable, **kw)
    out64, ls64, gr64 = orc.loss_and_grads(g.sd, g.hp, g.raw(), trainable, dtype=torch.float64, **kw)
    assert all(v.dtype == torch.float64 for v in out64.values()) and all(v.dtype == torch.float64 for v in gr64.values())
    for k in g.out:
        np.testing.assert_allclose(out32[k].detach().numpy(), out64[k].detach().numpy(), rtol=2e-5, atol=1e-4, err_msg=k)
    for k in g.loss:
        np.testing.assert_allclose(ls32[k].detach().numpy(), ls64[k].detach().numpy(), rtol=2e-5, atol=1e-4, err_msg=k)
    for k in trainable:
        want = gr64[k].numpy()
        scale = max(1.0, float(np.abs(want).max()))
        np.testing.assert_allclose(gr32[k].numpy(), want, rtol=1e-3, atol=2e-5 * scale, err_msg=k)
