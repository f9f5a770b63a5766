"""The split haplotype-CNN forward (hap_cnn_tc_kernel over the head layers, then hap_cnn_tail_kernel over the tail) against
the float64 oracle's haplotype CNN and against the single-kernel forward (PMT_CNN_SINGLE=1).  The library picks the pair
once the head kernel has a group of 16 variants for every SM (2 368 variants on 148 SMs); PMT_CNN_SINGLE=0 selects it at
any batch size, so that partial head groups and tail tiles are tested at every count.

Inside the tensor-core envelope every CNN ends in a Linear whose flattened input is at most 8 positions, so every such
shape has a tail: at v0.4.0 the last conv (6 positions in, 2 out, pool 2) and the Linear; with the last conv removed, the
Linear alone over 6 positions.  Haplotypes of 25 and 32 bases run the SIMT kernel.  Variant counts cover partial head
groups (16 variants) and partial tail tiles (128 variants)."""
import os

import numpy as np
import pytest
import torch

from helpers import batch_from_raw
from model_shapes import BY_NAME, V040_CNN, Shape, build_model
from oracle import artifact_oracle as orc
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.synthetic import make_arrays

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
F64 = torch.float64
V040 = Shape("v040")
LINEAR_TAIL = Shape("linear_tail", dict(ref_seq_layer_strings=V040_CNN[:9] + V040_CNN[12:]))   # flatten keeps 6 positions
SIZES = [1, 15, 16, 17, 127, 128, 129, 5000, 1_250_000]
TOL = {"tf32x3": 2e-5, "tf32": 5e-3}     # test_tensor_core_gpu.py's bounds on the sequence embedding


@pytest.fixture(autouse=True)
def _restore():
    yield
    L.set_precision("fp32")
    os.environ.pop("PMT_CNN_SINGLE", None)


def _raw(shape, n, seed):
    """n variants of one ref and one alt read (the CNN reads only the haplotypes), every code at every position."""
    rng = np.random.default_rng(seed)
    ones = np.ones(n, np.int64)
    ia, fa, reads = make_arrays(ones, ones, rng, n_info=shape.n_info, hap_len=shape.hap_len, row_bytes=shape.row_bytes)
    ia[:, 16:] = rng.integers(0, 5, ia[:, 16:].shape)
    return dict(reads_u8=reads, read_indices=None, ref_counts=ones, alt_counts=ones, info=fa[:, 6:].astype(np.float32),
                haplotypes=ia[:, 16:], labels=ia[:, 2].astype(np.int64), sources=np.zeros(n, np.int64))


def _oracle_seq_emb(model, shape, haps):
    """The float64 oracle's haplotype CNN, on the GPU in slices of 250 000 variants."""
    sd = {k: v.detach().to(DEV, F64) for k, v in model.state_dict().items() if k.startswith("haplotypes_cnn.")}
    out = []
    with torch.no_grad():
        for i in range(0, len(haps), 250_000):
            x = orc.one_hot_haplotypes(torch.as_tensor(haps[i:i + 250_000]), F64).to(DEV)
            out.append(orc.haplotype_cnn(sd, "haplotypes_cnn", shape.hp["ref_seq_layer_strings"], x).cpu())
    return torch.cat(out).numpy()


def _cnn_kernels(model, batch):
    """Names of the haplotype-CNN kernels one inference call launches."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        with torch.inference_mode():
            engine.forward_call(model.descriptor(), model.flat_weights(), batch)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "hap_cnn" in e.name}
    return {k for k in ("hap_cnn_tc_kernel", "hap_cnn_tail_kernel", "hap_cnn_kernel") if any(k + "<" in n or k + "(" in n for n in names)}


def _info_seq(model, batch, single=False, poison_tail=False):
    os.environ["PMT_CNN_SINGLE"] = "1" if single else "0"
    try:
        if not poison_tail:
            with torch.inference_mode():
                return engine.forward_call(model.descriptor(), model.flat_weights(), batch)["info_seq"].cpu()
        # a private workspace whose tail buffer (the last region of the forward's layout) holds NaN bytes
        import ctypes
        desc = model.descriptor()
        need = L.load().pmt_workspace_size(ctypes.byref(desc), ctypes.byref(batch.pmt_batch()), 0)
        tail = (batch.size() + 127) // 128 * 128 * 192 * 4
        ws = torch.zeros(need, dtype=torch.uint8, device=DEV)
        ws[need - 1024 - tail:] = 255
        with engine.use_workspace(DEV, ws), torch.inference_mode():
            return engine.forward_call(desc, model.flat_weights(), batch)["info_seq"].cpu()
    finally:
        os.environ.pop("PMT_CNN_SINGLE", None)


@pytest.mark.parametrize("shape", [V040, LINEAR_TAIL, BY_NAME["hap_50"], BY_NAME["hap_64"]], ids=lambda s: s.name)
def test_kernel_choice(shape):
    model = build_model(shape, DEV)
    small, large = (batch_from_raw(_raw(shape, n, 1), DEV) for n in (300, 5000))
    pair, single = {"hap_cnn_tc_kernel", "hap_cnn_tail_kernel"}, {"hap_cnn_tc_kernel"}
    for mode in ("tf32x3", "tf32"):
        L.set_precision(mode)
        if shape.cnn_tc:
            assert _cnn_kernels(model, large) == pair, mode
            assert _cnn_kernels(model, small) == single, mode       # fewer head groups than SMs
            os.environ["PMT_CNN_SINGLE"] = "1"
            assert _cnn_kernels(model, large) == single, mode
            os.environ["PMT_CNN_SINGLE"] = "0"
            assert _cnn_kernels(model, small) == pair, mode
            os.environ.pop("PMT_CNN_SINGLE")
        else:
            assert _cnn_kernels(model, large) == {"hap_cnn_kernel"}, mode
            assert _cnn_kernels(model, small) == {"hap_cnn_kernel"}, mode


@pytest.mark.parametrize("n", SIZES)
def test_split_forward_against_the_oracle_and_the_single_kernel(n):
    model = build_model(V040, DEV)
    raw = _raw(V040, n, 100 + n)
    batch = batch_from_raw(raw, DEV)
    d_info = model.descriptor().d_info
    want = _oracle_seq_emb(model, V040, raw["haplotypes"])
    for mode in ("tf32x3", "tf32"):
        L.set_precision(mode)
        split = _info_seq(model, batch, poison_tail=True)
        single = _info_seq(model, batch, single=True)
        assert torch.isfinite(split).all(), mode
        err = float(np.abs(split[:, d_info:].numpy() - want).max())
        print(f"[n={n} {mode}] split - oracle {err:.2e}")
        assert err <= TOL[mode], (mode, err)
        # the dense tail sums the shifted taps' products in their order (plus exact zeros): the single kernel's bits
        assert torch.equal(split, single), (mode, float((split - single).abs().max()))


def test_linear_only_tail_against_the_oracle():
    model = build_model(LINEAR_TAIL, DEV)
    raw = _raw(LINEAR_TAIL, 5000, 7)
    batch = batch_from_raw(raw, DEV)
    d_info = model.descriptor().d_info
    want = _oracle_seq_emb(model, LINEAR_TAIL, raw["haplotypes"])
    for mode in ("tf32x3", "tf32"):
        L.set_precision(mode)
        got = _info_seq(model, batch)[:, d_info:].numpy()
        err = float(np.abs(got - want).max())
        print(f"[linear tail {mode}] split - oracle {err:.2e}")
        assert err <= TOL[mode], (mode, err)


@pytest.mark.parametrize("dtype", [torch.int16, torch.int64])
@pytest.mark.parametrize("extra", [0, 9])
def test_haplotype_encodings(dtype, extra):
    """int16 / int64 haplotypes at the tight stride and with a gap: the split forward's bits equal the product batch's."""
    from test_batch_encodings_gpu import Recoded
    model = build_model(V040, DEV)
    raw = _raw(V040, 5000, 3)
    batch = batch_from_raw(raw, DEV)
    L.set_precision("tf32x3")
    want = _info_seq(model, batch)
    got = _info_seq(model, Recoded(batch, haps=(dtype, 2 * V040.hap_len + extra)))
    assert torch.equal(got, want)
