"""The read path, info MLP and haplotype CNN at model shapes other than v0.4.0, against the float64 oracle.

Every shape comes from model_shapes.py: the corners of the tensor-core envelope (max: d_read 31, d_info + d_seq 32, H 11,
E 16, K 6; min: d_model 16, H 2, one block, E 2, K 1; 12 blocks of odd widths with two sources; E 1), the SIMT kernels'
limits (d_model 64, E 32, K 14), one past each edge of the tensor-core envelope, the info MLP's three kernels and
haplotype lengths the tensor-core CNN does not take.  Each test first asserts which kernels run, so a shape that drops to
a fall-back fails instead of passing on other kernels.  The contracts are those the rest of the suite states."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import batch_from_raw
from model_shapes import BY_NAME, EDGE_SHAPES, HAP_SHAPES, INFO_SHAPES, SIMT_SHAPES, TC_SHAPES, build_model, long_set_raw, make_raw
from oracle import artifact_oracle as orc
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.utils.enums import Epoch
from test_backward_tc_gpu import _violations

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
F64 = torch.float64
SIZES = [300, 5000]          # either side of the 4 096-variant switch of the info MLP (warp kernel / rows kernel)
LONG_SHAPES = [(7, 3), (125, 3), (700, 300), (10, 15), (0, 200), (130, 1), (3, 1), (257, 255), (9, 2), (2900, 1500), (128, 128),
               (129, 1)]
ids = lambda s: s.name


@pytest.fixture(autouse=True)
def _restore():
    yield
    L.set_precision("fp32")


class Case:
    """A model of one shape, a batch (the product Batch of `raw` unless one is given), and the float64 oracle's outputs (and
    gradients) on it."""

    _oracle = {}    # (shape, batch key, grads) -> the float64 results, shared by the tests of both precision modes

    def __init__(self, shape, raw, grads=False, key=None, batch=None):
        self.shape, self.raw = shape, raw
        self.model = build_model(shape, DEV)
        self.batch = batch_from_raw(raw, DEV) if batch is None else batch
        self.sd = {k: v.detach().cpu() for k, v in self.model.state_dict().items()}
        self.names = [n for n, _ in self.model.named_parameters()]
        self.kw = dict(num_sources=shape.num_sources, source_adversarial_strength=0.3)
        cache_key = (shape.name, key, grads) if key is not None else None
        if cache_key in Case._oracle:
            self.want, self.want_losses, self.want_grads = Case._oracle[cache_key]
            return
        self.want_losses = self.want_grads = None
        if grads:
            self.want, self.want_losses, g = orc.loss_and_grads(self.sd, shape.hp, raw, self.names, dtype=F64, **self.kw)
            self.want = {k: v.detach() for k, v in self.want.items()}
            self.want_grads = {k: v.numpy() for k, v in g.items()}
        else:
            with torch.no_grad():
                self.want = orc.forward(self.sd, shape.hp, raw, dtype=F64)
        if cache_key is not None:
            Case._oracle[cache_key] = (self.want, self.want_losses, self.want_grads)

    def assert_kernels(self, mode):
        """The backward kernels and the saved-forward path this shape gets in `mode` (pmt_backward_kernels,
        pmt_train_saved_bytes): what model_shapes.py documents."""
        L.set_precision(mode)
        desc = self.model.descriptor()
        tc = mode != "fp32"
        assert L.backward_kernels(desc) == {"reads_tc": tc and self.shape.bwd_tc, "cnn_tc": tc and self.shape.cnn_tc}
        saved = L.load().pmt_train_saved_bytes(ctypes.byref(desc), ctypes.byref(self.batch.pmt_batch()))
        assert (saved > 0) == (mode == "tf32x3" and self.shape.bwd_tc and self.shape.cnn_tc), saved

    def assert_not_saturated(self):
        """The reference logits straddle zero and most sit well inside the tanh, so a wrong kernel cannot hide there."""
        lg = self.want["logits_b"].numpy()
        assert 0.1 <= np.mean(lg > 0) <= 0.9, np.mean(lg > 0)
        assert np.mean(np.abs(lg) < orc.MAX_LOGIT / 2) >= 0.4

    def forward(self, mode):
        self.assert_kernels(mode)
        self.model.set_epoch_type(Epoch.VALID)
        with torch.inference_mode():
            out = self.model.compute_batch_output(self.batch)
            info_seq = engine.forward_call(self.model.descriptor(), self.model.flat_weights(), self.batch)["info_seq"]
        torch.cuda.synchronize()
        return out, info_seq.cpu()

    def backward(self, mode):
        self.assert_kernels(mode)
        self.model.set_epoch_type(Epoch.TRAIN)
        for p in self.model.parameters():
            p.grad = None
        out = self.model.compute_batch_output(self.batch)
        losses = self.model.compute_batch_losses(out, self.batch)
        losses.total_loss.backward()
        grads = {n: (p.grad.detach().cpu().numpy() if p.grad is not None else np.zeros(tuple(p.shape), np.float32))
                 for n, p in self.model.named_parameters()}
        return out, losses, grads


def _report(case, what, errs):
    print(f"[{case.shape.name} B={len(case.raw['ref_counts'])}] {what}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))


def _err(got, want, rtol=0.0):
    """Largest |got - want| - rtol |want| (what an assert_close with this rtol compares with atol)."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.max(np.abs(got - want) - rtol * np.abs(want)))


def _check_forward(case, mode, logits_b_of_bk=0.0):
    """The forward against float64 under the suite's contracts; `logits_b_of_bk` widens logits_b's 1e-3 by that fraction
    of each variant's largest |logits_bk| (the log-likelihoods it is a difference of)."""
    out, info_seq = case.forward(mode)
    w = {k: v.numpy() for k, v in case.want.items() if isinstance(v, torch.Tensor)}
    d_info = case.model.descriptor().d_info
    got = dict(logits_b=out.logits_b.cpu().numpy(), logits_bk=out.logits_bk.cpu().numpy(),
               features_be=out.features_be.cpu().numpy(), ref_features_be=out.ref_features_be.cpu().numpy(),
               outlier_binary_logits=out.outlier_binary_logits.cpu().numpy(), info_seq=info_seq.numpy())
    if mode == "tf32":      # plain TF32 through ~45 layers: its stated 0.25 logit bound, signs away from zero
        err = _err(got["logits_b"], w["logits_b"])
        _report(case, mode, {"logits_b": err})
        assert err <= 0.25
        far = np.abs(w["logits_b"]) > 0.5
        assert np.array_equal(np.sign(got["logits_b"][far]), np.sign(w["logits_b"][far]))
        return out
    contract = dict(logits_b=(0, 1e-3), logits_bk=(5e-5, 2e-3), features_be=(1e-4, 2e-4), ref_features_be=(1e-4, 2e-4),
                    outlier_binary_logits=(5e-5, 2e-3))
    errs = {k: _err(got[k], w[k], rtol) for k, (rtol, _) in contract.items()}
    slack = logits_b_of_bk * np.abs(w["logits_bk"]).max(axis=1)
    errs["logits_b"] = float(np.max(np.abs(got["logits_b"] - w["logits_b"]) - slack))
    errs["info"] = _err(got["info_seq"][:, :d_info], w["info_seq_be"][:, :d_info], 2e-5)
    errs["seq_emb"] = _err(got["info_seq"][:, d_info:], w["ref_seq_emb"])
    _report(case, mode, errs)
    for k, (rtol, atol) in contract.items():
        if k == "logits_b" and logits_b_of_bk:
            assert errs[k] <= atol, f"{mode} logits_b {errs[k]:.3e} beyond {logits_b_of_bk:g} of max |logits_bk|"
            continue
        np.testing.assert_allclose(got[k], w[k], rtol=rtol, atol=atol, err_msg=f"{mode} {k}")
    np.testing.assert_allclose(got["info_seq"][:, :d_info], w["info_seq_be"][:, :d_info], rtol=2e-5, atol=2e-5, err_msg=f"{mode} info")
    np.testing.assert_allclose(got["info_seq"][:, d_info:], w["ref_seq_emb"], rtol=0, atol=2e-5, err_msg=f"{mode} seq emb")
    return out


def _check_gradients(case, mode):
    _, losses, got = case.backward(mode)
    for k in ("total_losses_b", "supervised_losses_b", "unsupervised_losses_b", "alt_count_losses_b", "source_prediction_losses_b"):
        np.testing.assert_allclose(getattr(losses, k).detach().cpu().numpy(), case.want_losses[k].detach().numpy(),
                                   rtol=2e-4, atol=2e-3, err_msg=k)
    want = case.want_grads
    if mode != "fp32" and case.shape.bwd_tc:    # tensor-core backward: 4e-3 of each tensor's max (one-entry: of their module's)
        bad = _violations(got, want)
        worst = max(float(np.abs(got[n] - w).max()) / max(float(np.abs(w).max()), 1e-3) for n, w in want.items() if w.size >= 8)
    else:                   # FP32 SIMT backward: 2e-3 of each tensor's max
        rel = {n: float(np.abs(got[n] - w).max()) / max(float(np.abs(w).max()), 1e-3) for n, w in want.items()}
        bad = sorted(((e, n) for n, e in rel.items() if e > 2e-3), reverse=True)
        worst = max(rel.values())
    _report(case, f"{mode} gradients", {"worst relative-to-max": worst})
    assert not bad, f"{mode} gradient error too large:\n" + "\n".join(f"{e:.3e} {n}" for e, n in bad[:25])
    cnn = [n for n in case.names if n.startswith("haplotypes_cnn")]
    assert all(np.abs(got[n]).max() > 0 for n in cnn)


# ---- the corners of the tensor-core envelope ----
@pytest.mark.parametrize("n_variants", SIZES)
@pytest.mark.parametrize("shape", TC_SHAPES, ids=ids)
def test_tensor_core_shapes_forward_against_float64(shape, n_variants):
    case = Case(shape, make_raw(shape, n_variants, seed=n_variants))
    case.assert_not_saturated()
    for mode in ("tf32x3", "fp32", "tf32"):
        _check_forward(case, mode)


# pmt_backward needs the FP32 read-path backward's shared-memory plan (bwd_smem_bytes in pmt_backward.cu: the model's
# weight and activation stages, the set sums of 2 x 128 reads and the head's accumulators) to fit in 227 KB, in every
# precision mode: that kernel also takes the sets longer than a tile.  Shapes with trains=False in model_shapes.py are
# past it (the max corner, H 12, the SIMT limits): every backward refuses, whatever the batch.
TOO_WIDE = "shared-memory plan"


# reducer._model.0.alpha of the 12-block model on these 5 000 variants is a sum whose terms cancel 8 000-fold
# (sum |W U| + |b Ub| over |<W, U> + <b, Ub>| in the float64 oracle; 20-1 000 elsewhere): the TF32 operands of the
# tensor-core backward leave it 2e-2 off against its module's largest one-entry gradient (contract 4e-3).  The fp32 mode
# meets 2e-3 on the same case.
ILL_CONDITIONED = pytest.mark.xfail(strict=True, reason="one-entry gradient cancelling 8 000-fold, beyond TF32 operands")


def _gradient_params():
    for shape in TC_SHAPES:
        for n in SIZES:
            for mode in ("tf32x3", "fp32"):
                marks = [ILL_CONDITIONED] if (shape.name, n, mode) == ("deep_odd", 5000, "tf32x3") else []
                yield pytest.param(shape, n, mode, id=f"{shape.name}-{n}-{mode}", marks=marks)


@pytest.mark.parametrize("shape,n_variants,mode", list(_gradient_params()))
def test_tensor_core_shapes_gradients_against_float64(shape, n_variants, mode):
    """The max corner cannot train in either mode (TOO_WIDE)."""
    case = Case(shape, make_raw(shape, n_variants, seed=10 + n_variants), grads=shape.trains, key=n_variants)
    if not shape.trains:
        with pytest.raises(RuntimeError, match=TOO_WIDE):
            case.backward(mode)
        return
    _check_gradients(case, mode)


@pytest.mark.parametrize("shape", [s for s in TC_SHAPES if s.trains and s.bwd_tc], ids=ids)
def test_saved_forward_equals_recompute_at_other_step_programs(shape, monkeypatch):
    """The saved-forward buffer and the backward workspace (their maps in pmt_call.cu) are sized from the step
    program: outputs and gradients of the saved forward are BITWISE those of the recompute, which here walks the tile list
    in several ranges, and both are bitwise reproducible."""
    monkeypatch.setenv("PMT_BWD_CHUNK_TILES", "64")
    case = Case(shape, make_raw(shape, 5000, seed=77))

    def run():
        out, _, grads = case.backward("tf32x3")
        return {k: getattr(out, k).detach().cpu().numpy() for k in ("logits_b", "logits_bk", "features_be", "ref_features_be")}, grads

    saved = run()
    monkeypatch.setenv("PERMUTECT_B200_TRAIN_SAVED", "0")
    recompute = run()
    recompute2 = run()
    monkeypatch.delenv("PERMUTECT_B200_TRAIN_SAVED")
    saved2 = run()
    for other in (recompute, recompute2, saved2):
        for a, b in zip(saved, other):
            assert a.keys() == b.keys()
            for k in a:
                np.testing.assert_array_equal(a[k], b[k], err_msg=k)


# ---- sets longer than a tile at the max corner and at 12 blocks ----
@pytest.mark.parametrize("shape", [BY_NAME["max_corner"], BY_NAME["deep_odd"]], ids=ids)
def test_long_sets_against_float64(shape, monkeypatch):
    """Sets of up to 4 400 reads among tile-sized ones: the tensor-core long-set kernel (single-side tiles meeting through
    global memory, pmt_tc.cuh: LongTile) and the FP32 long-set kernel (PMT_LONG_SIMT=1), both against float64; the
    tensor-core one bitwise reproducible."""
    case = Case(shape, long_set_raw(shape, LONG_SHAPES, seed=11))
    outs = {}
    for simt in ("0", "1"):
        monkeypatch.setenv("PMT_LONG_SIMT", simt)
        outs[simt] = _check_forward(case, "tf32x3")
    torch.testing.assert_close(outs["0"].logits_b, outs["1"].logits_b, rtol=0, atol=1e-3)
    # split-precision TF32 and FP32 FMA do not round alike: equal bits would mean both runs took the same (SIMT) kernel
    assert not torch.equal(outs["0"].logits_bk, outs["1"].logits_bk)
    monkeypatch.setenv("PMT_LONG_SIMT", "0")
    again, _ = case.forward("tf32x3")
    for name in ("logits_b", "logits_bk", "features_be", "ref_features_be"):
        assert torch.equal(getattr(outs["0"], name), getattr(again, name)), name


@pytest.mark.parametrize("shape", [BY_NAME["max_corner"], BY_NAME["deep_odd"]], ids=ids)
def test_mixed_long_and_tile_sized_sets_gradients_against_float64(shape):
    """Sets longer than a tile keep the FP32 long-set backward; the tile-sized sets around them take the tensor cores."""
    sets = [(7, 3), (125, 3), (300, 100), (10, 15), (0, 20), (130, 1), (3, 1), (9, 2), (0, 1), (40, 60)]
    case = Case(shape, long_set_raw(shape, sets, seed=12), grads=shape.trains)
    if not shape.trains:
        with pytest.raises(RuntimeError, match=TOO_WIDE):
            case.backward("tf32x3")
        return
    _check_gradients(case, "tf32x3")
    _, _, a = case.backward("tf32x3")
    _, _, b = case.backward("tf32x3")
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


# ---- the SIMT kernels' limits ----
@pytest.mark.parametrize("shape", SIMT_SHAPES, ids=ids)
def test_simt_limits_against_float64(shape):
    case = Case(shape, make_raw(shape, 300, seed=5))
    case.assert_not_saturated()
    _check_forward(case, "fp32")
    with pytest.raises(RuntimeError, match=TOO_WIDE):     # see TOO_WIDE
        case.backward("fp32")


# ---- one past each edge of the tensor-core envelope ----
@pytest.mark.parametrize("shape", EDGE_SHAPES, ids=ids)
def test_one_past_each_edge(shape):
    """The FP32 kernels take the shape and meet the contract; the tensor-core forward refuses it loudly, the backward
    reports the SIMT read path and the training forward has no saved path."""
    grads = shape.name == "d_read_32"
    case = Case(shape, make_raw(shape, 300, seed=6), grads=grads)
    case.assert_not_saturated()
    _check_forward(case, "fp32")
    if not shape.trains:
        with pytest.raises(RuntimeError, match=TOO_WIDE):
            case.backward("fp32")
    elif grads:
        _check_gradients(case, "fp32")
    case.assert_kernels("tf32x3")
    case.model.set_epoch_type(Epoch.VALID)
    with pytest.raises(RuntimeError, match="envelope"), torch.inference_mode():
        case.model.compute_batch_output(case.batch)


# ---- the info MLP's kernels ----
@pytest.mark.parametrize("n_variants", SIZES)
@pytest.mark.parametrize("shape", INFO_SHAPES, ids=ids)
def test_info_mlp_shapes_against_float64(shape, n_variants):
    case = Case(shape, make_raw(shape, n_variants, seed=20 + n_variants))
    case.assert_not_saturated()
    for mode in ("fp32", "tf32x3") if shape.reads_tc else ("fp32",):
        _check_forward(case, mode)


@pytest.mark.parametrize("shape", [BY_NAME["info_w32"], BY_NAME["n_info_9"], BY_NAME["n_info_128"]], ids=ids)
def test_info_warp_and_rows_kernels_are_bitwise_equal(shape):
    """info_mlp_warp_kernel (batches up to 4 096 variants) and info_mlp_rows_kernel (larger ones) sum in the same order:
    the same 4 096 variants alone and as the head of a 4 097-variant batch give the same bits."""
    raw = make_raw(shape, 4097, seed=31)
    model = build_model(shape, DEV)
    model.set_epoch_type(Epoch.VALID)
    L.set_precision("fp32")
    desc = model.descriptor()
    head = {k: (v[:4096] if k in ("ref_counts", "alt_counts", "info", "haplotypes", "labels", "sources") else v) for k, v in raw.items()}
    head["reads_u8"] = np.concatenate((raw["reads_u8"][:int(raw["ref_counts"][:4096].sum())],
                                       raw["reads_u8"][int(raw["ref_counts"].sum()):int(raw["ref_counts"].sum()) + int(raw["alt_counts"][:4096].sum())]))
    with torch.inference_mode():
        alone = engine.forward_call(desc, model.flat_weights(), batch_from_raw(head, DEV))["info_seq"][:, :desc.d_info].cpu()
        whole = engine.forward_call(desc, model.flat_weights(), batch_from_raw(raw, DEV))["info_seq"][:4096, :desc.d_info].cpu()
    assert torch.equal(alone, whole)


# ---- haplotype lengths outside the tensor-core CNN ----
@pytest.mark.parametrize("shape", HAP_SHAPES, ids=ids)
def test_haplotype_lengths_against_float64(shape):
    case = Case(shape, make_raw(shape, 300, seed=40), grads=True)
    case.assert_not_saturated()
    for mode in ("tf32x3", "fp32"):
        _check_forward(case, mode)
        _check_gradients(case, mode)
