"""The model kernels on every batch encoding the C-ABI accepts (include/permutect_b200.h: PmtBatch), against the float64
oracle and against the product batch.

The product batch (data/batch.py) has one layout: compressed uint8 rows of 12 bytes, fp16 info at stride I + 6, int16
haplotypes at stride 2L + 16, an exact row count.  The kernels branch on each part of it:
  * compressed rows of 7..15 bytes (F = 56..64): the tensor-core read kernels fetch rows through their meta warp only at 12
    bytes and take F <= 61; the SIMT decode takes any width;
  * decoded rows (PMT_READS_F32 / F16): the tensor-core forward adds layer 0's low-half pass, which only arbitrary fp32 reads
    need -- decoded compressed rows (bits and k/32) are exact in TF32;
  * info in fp16 or fp32 at any stride and base: the warp (<= 4 096 variants), rows and tile-GEMM info kernels, and the rows
    kernel's raw fp16 copy (fp16, stride I..I+8, 4-byte aligned base);
  * haplotypes in int16 or int64 at any stride: every haplotype-CNN forward and backward kernel;
  * n_rows <= 0 ("unknown") or over-estimated, max_rows_per_variant over-estimated: grid sizes, the tile-count bound of the
    tensor-core training path and the long-set layout.
Each test first asserts which kernels run, so a fall-back fails instead of passing on other kernels.  The contracts are
those the rest of the suite states; encodings of equal values give bitwise-equal results within one precision mode."""
import numpy as np
import pytest
import torch

from helpers import batch_from_raw
from model_shapes import BY_NAME, Shape, build_model, long_set_raw, make_raw
from oracle import artifact_oracle as orc
from permutect_b200.data.batch import DownsampledBatch
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.utils.enums import Epoch
from test_head_backward_gpu import check_against_oracle, gradients, head_names
from test_model_shapes_gpu import DEV, LONG_SHAPES, Case, _check_forward, _check_gradients, _report

pytestmark = pytest.mark.gpu
V040 = Shape("v040")
# the model seed of each width: logits of both signs, mostly far from saturation, on make_raw(shape, 300, seed=row_bytes)
ROW_SEEDS = {7: 1, 9: 8, 11: 0, 12: 0, 13: 0, 15: 1}
TC_ROWS, WIDE_ROWS = [7, 9, 11, 12], [13, 15]
OUT_NAMES = ("logits_b", "logits_bk", "features_be", "ref_features_be", "outlier_binary_logits")


def rows_shape(row_bytes):
    return Shape(f"rows_{row_bytes}", n_read_features=row_bytes + 49, seed=ROW_SEEDS[row_bytes], reads_tc=row_bytes <= 12)


@pytest.fixture(autouse=True)
def _restore():
    yield
    L.set_precision("fp32")


class Recoded:
    """A product Batch as the C-ABI sees it with another encoding or other hints: its PmtBatch points info and haplotypes
    at copies owned here (`info` = (dtype, stride, base offset in elements), `haps` = (dtype, stride)), or carries another
    n_rows / max_rows_per_variant.  Stride gaps hold valid values, which a kernel reading the wrong columns would pick up."""

    def __init__(self, batch, info=None, haps=None, n_rows=None, max_rows=None):
        self.batch, self.reads = batch, batch.reads
        self.n_rows, self.max_rows = n_rows, max_rows
        self.info = self.haps = None
        B = batch.size()
        if info is not None:
            dtype, stride, offset = info
            x = batch.get_info_be()
            buf = torch.full((offset + B * stride,), 7.0, dtype=dtype, device=x.device)
            buf[offset:].view(B, stride)[:, :x.shape[1]] = x.to(dtype)
            self.info = (buf, buf.data_ptr() + offset * buf.element_size(), stride, L.F16 if dtype == torch.float16 else L.F32)
        if haps is not None:
            dtype, stride = haps
            h = batch.get_haplotypes_bs()
            buf = torch.full((B, stride), 3, dtype=dtype, device=h.device)
            buf[:, :h.shape[1]] = h.to(dtype)
            self.haps = (buf, stride, L.I16 if dtype == torch.int16 else L.I64)

    def size(self):
        return self.batch.size()

    def pmt_batch(self):
        pb = self.batch.pmt_batch()
        if self.info is not None:
            _, pb.info, pb.info_stride, pb.info_kind = self.info
        if self.haps is not None:
            buf, pb.hap_stride, pb.hap_kind = self.haps
            pb.haplotypes = buf.data_ptr()
        if self.n_rows is not None:
            pb.n_rows = self.n_rows
        if self.max_rows is not None:
            pb.max_rows_per_variant = self.max_rows
        return pb


def _calls(model, batch, mode):
    """Inference forward, training forward and backward (seeded upstream gradients) straight through the C-ABI calls."""
    L.set_precision(mode)
    desc = model.descriptor()
    B = batch.size()
    gen = torch.Generator().manual_seed(B)
    g = [torch.randn(shape, generator=gen).to(DEV) for shape in ((B, desc.n_clusters + 2), (B, desc.d_feat), (B, desc.d_feat))]
    with torch.no_grad():
        flat = model.flat_weights()
        out = engine.forward_call(desc, flat, batch)
        train = engine.forward_call(desc, flat, batch, for_training=True)
        d_flat = engine.backward_call(desc, flat, batch, *g, train["info_seq"], train.get("saved"))
    got = {k: out[k] for k in ("logits_bk", "logits_b", "outlier_logits", "alt_means", "ref_means", "info_seq")}
    got.update({"train " + k: train[k] for k in ("logits_bk", "alt_means", "ref_means", "info_seq")})
    got["d_flat"] = d_flat
    got = {k: v.cpu() for k, v in got.items()}
    got["saved"] = "saved" in train
    return got


def _assert_bitwise(got, want, what):
    assert got.keys() == want.keys()
    for k in want:
        if isinstance(want[k], torch.Tensor):
            assert torch.equal(got[k], want[k]), f"{what}: {k} differs by {float((got[k] - want[k]).abs().max()):.3e}"
        else:
            assert got[k] == want[k], (what, k)


def _outputs(out):
    return {k: getattr(out, k).detach().cpu() for k in OUT_NAMES}


def _max_diff(a, b):
    return max(float((a[k] - b[k]).abs().max()) for k in a)


# ---- compressed rows of 7..15 bytes ----
@pytest.mark.parametrize("row_bytes", TC_ROWS)
def test_read_row_widths_forward_against_float64(row_bytes):
    """Rows of other than 12 bytes take the per-byte decode of the tensor-core forward and the SIMT tile_decode."""
    shape = rows_shape(row_bytes)
    case = Case(shape, make_raw(shape, 300, seed=row_bytes))
    assert case.batch.reads.shape[1] == row_bytes
    case.assert_not_saturated()
    for mode in ("tf32x3", "fp32", "tf32"):
        _check_forward(case, mode)


@pytest.mark.parametrize("row_bytes", TC_ROWS)
def test_read_row_widths_gradients_against_float64(row_bytes, monkeypatch):
    """tf32x3 through the saved training forward and through the recompute, then the FP32 kernels."""
    shape = rows_shape(row_bytes)
    case = Case(shape, make_raw(shape, 300, seed=10 + row_bytes), grads=True, key=300)
    print("saved training forward:")
    _check_gradients(case, "tf32x3")      # Case.assert_kernels: the saved forward exists for this batch
    monkeypatch.setenv("PERMUTECT_B200_TRAIN_SAVED", "0")
    print("recompute:")
    _check_gradients(case, "tf32x3")
    monkeypatch.delenv("PERMUTECT_B200_TRAIN_SAVED")
    _check_gradients(case, "fp32")


@pytest.mark.parametrize("row_bytes", TC_ROWS)
def test_read_row_widths_head_backward_against_float64(row_bytes):
    """The trunk frozen, as in a calibration epoch: pmt_head_backward over the per-read features of the forward."""
    shape = rows_shape(row_bytes)
    case = Case(shape, make_raw(shape, 300, seed=10 + row_bytes), grads=True, key=300)
    trainable = head_names(case.model)
    for mode in ("fp32", "tf32x3"):
        got = gradients(case.model, case.batch, mode, trainable)
        assert case.model.trunk_frozen()
        check_against_oracle(case, got, trainable, mode, "head tensors")


# logits_b is a difference of the cluster log-likelihoods logits_bk, which reach 3.5e4 on the sets of hundreds of alt reads
# at this shape: it is held to 1e-3 plus 1e-6 of its variant's largest |logits_bk|, a few FP32 ulps of the terms it is the
# difference of (the FP32 oracle itself is 3.5e-4 off float64 there; the kernels' other summation order, 3e-3).
LONG_LOGITS_B = 1e-6


def test_read_rows_of_7_bytes_in_sets_longer_than_a_tile(monkeypatch):
    """The tensor-core long-set kernel and the FP32 one decode 7-byte rows too."""
    shape = rows_shape(7)
    case = Case(shape, long_set_raw(shape, LONG_SHAPES, seed=11))
    for simt in ("0", "1"):
        monkeypatch.setenv("PMT_LONG_SIMT", simt)
        _check_forward(case, "tf32x3", logits_b_of_bk=LONG_LOGITS_B)
    _check_forward(case, "fp32", logits_b_of_bk=LONG_LOGITS_B)


@pytest.mark.parametrize("row_bytes", WIDE_ROWS)
def test_read_rows_past_the_tensor_core_envelope(row_bytes):
    """F = 62 and 64: the FP32 kernels take them and meet the contract; the tensor-core forward refuses them loudly."""
    shape = rows_shape(row_bytes)
    case = Case(shape, make_raw(shape, 300, seed=row_bytes), grads=True)
    case.assert_not_saturated()
    _check_forward(case, "fp32")
    _check_gradients(case, "fp32")
    case.assert_kernels("tf32x3")
    case.model.set_epoch_type(Epoch.VALID)
    with pytest.raises(RuntimeError, match="envelope"), torch.inference_mode():
        case.model.compute_batch_output(case.batch)


# ---- decoded reads ----
@pytest.mark.parametrize("dtype", [np.float32, np.float16], ids=["f32", "f16"])
def test_decoded_reads_against_float64_and_the_compressed_rows(dtype):
    """The compressed rows decoded (bits and k/32: exact in fp16 and in TF32): the FP32 kernels give the compressed batch's
    bits; tf32x3 meets the contract."""
    case = Case(V040, make_raw(V040, 300, seed=30), grads=True, key="decoded")
    u8 = case.batch
    decoded = batch_from_raw(dict(case.raw, reads_u8=orc.decode_reads(case.raw["reads_u8"]).astype(dtype)), DEV)
    assert decoded.pmt_batch().reads_kind == (L.READS_F32 if dtype == np.float32 else L.READS_F16)
    for mode in ("fp32", "tf32x3"):
        case.batch = u8
        want_out, want_grads = _outputs(case.forward(mode)[0]), case.backward(mode)[2]
        case.batch = decoded
        got_out = _outputs(_check_forward(case, mode))
        _check_gradients(case, mode)
        got_grads = case.backward(mode)[2]
        grad_diff = max(float(np.abs(got_grads[n] - want_grads[n]).max()) for n in want_grads)
        _report(case, f"{mode} decoded {np.dtype(dtype).name} vs compressed",
                {"outputs": _max_diff(got_out, want_out), "gradients": grad_diff})
        if mode == "fp32":
            _assert_bitwise(got_out, want_out, "fp32 outputs")
            for n in want_grads:
                np.testing.assert_array_equal(got_grads[n], want_grads[n], err_msg=n)


def test_arbitrary_fp32_reads_against_float64():
    """Reads that are not TF32-exact: tf32x3 needs layer 0's low-half pass to meet its contract (the float64 oracle on the
    reads rounded to TF32 is 1e-2 off in the logits and 1e-3 in the features, against contracts of 1e-3 and 2e-4)."""
    raw = make_raw(V040, 300, seed=70)
    reads_f = (4 * np.random.default_rng(71).standard_normal((len(raw["reads_u8"]), 61))).astype(np.float32)
    assert np.mean(reads_f.view(np.uint32) & 0x1FFF != 0) > 0.99      # bits below TF32's 10-bit mantissa
    case = Case(V040, dict(raw, reads_u8=reads_f, reads_f=reads_f), grads=True)
    assert case.batch.pmt_batch().reads_kind == L.READS_F32
    case.assert_not_saturated()
    for mode in ("tf32x3", "fp32"):
        _check_forward(case, mode)
        _check_gradients(case, mode)
    _check_forward(case, "tf32")


def _downsample(raw, rng, keep=0.6):
    """Kept rows of each variant (batch order: every kept ref row, then every kept alt row; at least one alt row each)."""
    ref, alt = raw["ref_counts"], raw["alt_counts"]
    ref_start = np.concatenate(([0], np.cumsum(ref)[:-1]))
    alt_start = int(ref.sum()) + np.concatenate(([0], np.cumsum(alt)[:-1]))
    ref_idx, alt_idx = [], []
    for b in range(len(ref)):
        ka = np.flatnonzero(rng.random(alt[b]) < keep)
        ref_idx.append(ref_start[b] + np.flatnonzero(rng.random(ref[b]) < keep))
        alt_idx.append(alt_start[b] + (ka if len(ka) else np.zeros(1, np.int64)))
    idx = np.concatenate(ref_idx + alt_idx).astype(np.int64)
    return idx, np.array([len(i) for i in ref_idx], np.int64), np.array([len(i) for i in alt_idx], np.int64)


def test_downsampled_batch_of_decoded_reads():
    """read_indices gather decoded rows: against float64, and in FP32 bitwise the downsampled compressed batch."""
    raw = make_raw(V040, 300, seed=80)
    idx, ref_c, alt_c = _downsample(raw, np.random.default_rng(81))

    def downsampled(reads):
        parent = batch_from_raw(dict(raw, reads_u8=reads), DEV)
        return DownsampledBatch(parent, read_indices=torch.from_numpy(idx), ref_counts=torch.from_numpy(ref_c),
                                alt_counts=torch.from_numpy(alt_c))

    decoded = downsampled(orc.decode_reads(raw["reads_u8"]))
    assert decoded.read_indices is not None and decoded.pmt_batch().reads_kind == L.READS_F32
    case = Case(V040, dict(raw, read_indices=idx, ref_counts=ref_c, alt_counts=alt_c), grads=True, batch=decoded)
    outs = {}
    for mode in ("tf32x3", "fp32"):
        outs[mode] = _outputs(_check_forward(case, mode))
        _check_gradients(case, mode)
    case.batch = downsampled(raw["reads_u8"])
    _assert_bitwise(outs["fp32"], _outputs(case.forward("fp32")[0]), "fp32 decoded vs compressed, downsampled")


# ---- info and haplotype encodings ----
N_INFO_4 = Shape("n_info_4", n_info=4)
# (shape, variants): the warp and rows info kernels (either side of 4 096 variants), the tile-GEMM one, the SIMT CNN in
# every mode (hap_50), and 4 info features, where the rows kernel's raw fp16 tile is larger than its feature-major one
ENCODING_CASES = [(V040, 300), (V040, 5000), (BY_NAME["info_tile_gemm"], 300), (BY_NAME["hap_50"], 300), (N_INFO_4, 5000)]
INFO_STRIDES = {"I": lambda i: i, "I+6": lambda i: i + 6, "I+8": lambda i: i + 8, "I+9": lambda i: i + 9, "2I+3": lambda i: 2 * i + 3}
INFO_ENCODINGS = ([(torch.float16, s, 0) for s in INFO_STRIDES] + [(torch.float32, s, 0) for s in INFO_STRIDES]
                  + [(torch.float16, "I+6", 1)])          # a base one half past 4-byte alignment
HAP_ENCODINGS = [(torch.int16, 0), (torch.int64, 0), (torch.int16, 5), (torch.int64, 5)]     # stride 2L + this


@pytest.mark.parametrize("shape,n_variants", ENCODING_CASES, ids=[f"{s.name}-{n}" for s, n in ENCODING_CASES])
def test_info_and_haplotype_encodings_are_bitwise_equal(shape, n_variants):
    """fp16 and fp32 info at strides I, I+6, I+8, I+9, 2I+3 and at a misaligned base; int16 and int64 haplotypes at strides
    2L and 2L+5: the same values give the product batch's bits in the forward, the training forward and the backward, in
    FP32 and in tf32x3 (the tensor-core CNN, its SAVE variant and its backward)."""
    case = Case(shape, make_raw(shape, n_variants, seed=90 + n_variants))
    I, n_hap = case.raw["info"].shape[1], case.raw["haplotypes"].shape[1]
    for mode in ("fp32", "tf32x3"):
        _check_forward(case, mode)       # the product batch against float64, and the kernel choice
        want = _calls(case.model, case.batch, mode)
        assert want["saved"] == (mode == "tf32x3" and shape.bwd_tc and shape.cnn_tc)
        for i, (info_dtype, stride, offset) in enumerate(INFO_ENCODINGS):
            hap_dtype, hap_pad = HAP_ENCODINGS[i % len(HAP_ENCODINGS)]
            enc = Recoded(case.batch, info=(info_dtype, INFO_STRIDES[stride](I), offset), haps=(hap_dtype, n_hap + hap_pad))
            what = f"{mode} info {info_dtype} stride {stride} offset {offset}, haplotypes {hap_dtype} stride 2L+{hap_pad}"
            _assert_bitwise(_calls(case.model, enc, mode), want, what)
        _report(case, f"{mode} {len(INFO_ENCODINGS)} info / haplotype encodings", {"bitwise vs product batch": 0.0})


# ---- row hints ----
def _hint_raw(sets):
    if sets == "wgs":
        return make_raw(V040, 5000, seed=100)
    return long_set_raw(V040, [(30, 30)] * 1500, seed=101)     # two sets to a tile; 16 rows per variant is a quarter


@pytest.mark.parametrize("path", ["saved", "recompute", "fp32"])
@pytest.mark.parametrize("sets", ["wgs", "sixty"])
def test_row_hints_give_the_exact_hint_bits(sets, path, monkeypatch):
    """n_rows unknown (0, -1) or 3x the real count, max_rows_per_variant 3x the longest set (for 60-row sets: past a tile,
    so the long-set kernels are planned and find nothing): the forward, the training forward and the backward give the
    bits of the exact hints.  At these sizes every grid and planner claim is the same for all hints."""
    mode = "fp32" if path == "fp32" else "tf32x3"
    if path == "recompute":
        monkeypatch.setenv("PERMUTECT_B200_TRAIN_SAVED", "0")
    model = build_model(V040, DEV)
    batch = batch_from_raw(_hint_raw(sets), DEV)
    L.set_precision(mode)
    assert L.backward_kernels(model.descriptor()) == {"reads_tc": mode != "fp32", "cnn_tc": mode != "fp32"}
    rows, longest = int(batch.pmt_batch().n_rows), batch.max_rows_per_variant
    want = _calls(model, batch, mode)
    assert want["saved"] == (path == "saved")
    for n_rows, max_rows in ((0, None), (-1, None), (3 * rows, None), (None, 3 * longest), (0, 3 * longest)):
        _assert_bitwise(_calls(model, Recoded(batch, n_rows=n_rows, max_rows=max_rows), mode), want,
                        f"{path} n_rows {n_rows} max_rows_per_variant {max_rows}")
    print(f"[v040 {sets} B={batch.size()} rows={rows}] {path}: 5 row hints bitwise equal to the exact ones")
