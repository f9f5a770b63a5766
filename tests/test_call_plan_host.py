"""The call plan without a GPU: a call the kernels' envelopes rule out is refused before anything is enqueued, and the
sizes and backward kernels it answers with stay those it has always answered with."""
import ctypes

import pytest
import torch

from model_shapes import ALL_SHAPES, EDGE_SHAPES, SIMT_SHAPES, build_model
from permutect_b200.engine import library as L

CPU = torch.device("cpu")
OVERRIDES = ("PMT_CNN_SINGLE", "PMT_TC_PACKED", "PMT_LONG_SIMT", "PMT_BWD_CHUNK_TILES")
PLACEHOLDER = 0x100000   # never dereferenced: the call is refused first
MODES = ("fp32", "tf32x3", "tf32")


@pytest.fixture(autouse=True)
def _defaults(monkeypatch):
    for name in OVERRIDES:
        monkeypatch.delenv(name, raising=False)
    yield
    L.set_precision("fp32")


def _batch(n_variants, reads_per_variant, max_rows, n_rows=None):
    pb = L.PmtBatch()
    pb.n_variants = n_variants
    pb.n_rows = n_variants * reads_per_variant if n_rows is None else n_rows
    pb.total_ref, pb.max_rows_per_variant = -1, max_rows
    for name in ("reads", "ref_off", "alt_off", "info", "haplotypes"):
        setattr(pb, name, PLACEHOLDER)
    return pb


# Without a batch; a small one; one past the CNN head + tail threshold of v0.4.0 on 148 SMs (16-variant groups); one with
# sets longer than a tile; one without a row count.
BATCHES = (None, (64, 20, 40), (2369, 20, 40), (1000, 30, 400), (3000, 20, 60, 0))


def _sizes(lib, desc, batch):
    pb = None if batch is None else ctypes.byref(_batch(*batch))
    return (lib.pmt_workspace_size(ctypes.byref(desc), pb, 0), lib.pmt_workspace_size(ctypes.byref(desc), pb, 1),
            lib.pmt_train_saved_bytes(ctypes.byref(desc), pb) if pb is not None else 0)


@pytest.mark.skipif(torch.cuda.is_available(), reason="placeholder pointers must never reach a device")
@pytest.mark.parametrize("shape", SIMT_SHAPES + EDGE_SHAPES, ids=lambda s: s.name)
def test_tensor_core_forward_refuses_before_any_cuda_call(shape):
    """On a machine without a GPU any CUDA call fails, so the error shows which came first: the envelope check or the
    first memset."""
    desc = build_model(shape, CPU).descriptor()
    lib = L.load()
    L.set_precision("tf32x3")
    pb = _batch(1000, 25, 40)
    ws = lib.pmt_workspace_size(ctypes.byref(desc), ctypes.byref(pb), 0)
    assert ws > 0
    out = L.PmtOutputs(*([PLACEHOLDER] * len(L.PmtOutputs._fields_)))
    for fn in (lib.pmt_forward, lib.pmt_forward_prepared):
        rc = fn(ctypes.byref(desc), PLACEHOLDER, ctypes.byref(pb), ctypes.byref(out), PLACEHOLDER, ws, None)
        assert rc != 0
        assert b"tensor-core kernel's envelope" in lib.pmt_last_error(), lib.pmt_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="placeholder pointers must never reach a device")
@pytest.mark.parametrize("shape", [s for s in ALL_SHAPES if not s.trains], ids=lambda s: s.name)
def test_fp32_backward_refuses_before_any_cuda_call(shape):
    desc = build_model(shape, CPU).descriptor()
    lib = L.load()
    L.set_precision("fp32")
    pb = _batch(1000, 25, 40)
    ws = lib.pmt_workspace_size(ctypes.byref(desc), ctypes.byref(pb), 1)
    grads = L.PmtOutGrads(*([PLACEHOLDER] * 3 + [None, None]))
    rc = lib.pmt_backward(ctypes.byref(desc), PLACEHOLDER, ctypes.byref(pb), ctypes.byref(grads), PLACEHOLDER, PLACEHOLDER, ws, None)
    assert rc != 0
    assert b"shared-memory plan" in lib.pmt_last_error(), lib.pmt_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="placeholder pointers must never reach a device")
@pytest.mark.parametrize("base_offset", [None, 4, 256], ids=["one_byte_short", "base+4", "base+256"])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", ALL_SHAPES, ids=lambda s: s.name)
def test_buffers_are_resolved_before_any_cuda_call(shape, mode, base_offset):
    """pmt_forward, pmt_forward_train and pmt_backward lay the call plan's maps over their buffers before their first CUDA
    call.  One byte less than the size the library reports is refused with the size message.  At the exact size, from a
    base that is not aligned, every region realigns inside its slack and the call gets past the bounds check to that CUDA
    call, which fails on a machine without a GPU (unless the call plan refuses the call first)."""
    desc = build_model(shape, CPU).descriptor()
    lib = L.load()
    L.set_precision(mode)
    out = L.PmtOutputs(*([PLACEHOLDER] * len(L.PmtOutputs._fields_)))
    grads = L.PmtOutGrads(*([PLACEHOLDER] * 3 + [None, None]))
    short = 1 if base_offset is None else 0
    ws = PLACEHOLDER + (base_offset or 0)
    for batch in BATCHES[1:]:
        pb = _batch(*batch)
        fwd, bwd, saved = _sizes(lib, desc, batch)
        args = (ctypes.byref(desc), PLACEHOLDER, ctypes.byref(pb))
        calls = [lambda: lib.pmt_forward(*args, ctypes.byref(out), ws, fwd - short, None),
                 lambda: lib.pmt_backward(*args, ctypes.byref(grads), PLACEHOLDER, ws, bwd - short, None)]
        if saved:   # the saved buffer one byte short, or the workspace from the unaligned base
            calls.append(lambda: lib.pmt_forward_train(*args, ctypes.byref(out), ws, fwd, PLACEHOLDER, saved - short, None))
        for call in calls:
            assert call() != 0
            err = lib.pmt_last_error()
            if short:
                assert b"too small" in err, (batch, err)
            else:
                # past the resolver: the first CUDA call failed, or the plan refused the call after the buffers were resolved
                assert b"too small" not in err and b"ends past" not in err, (batch, err)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", ALL_SHAPES, ids=lambda s: s.name)
def test_sizes_and_backward_kernels_are_unchanged(shape, mode):
    """Forward and backward workspace and saved-forward bytes for each of BATCHES, then the backward kernels: the values
    the library gave before every kernel choice moved into the call plan (148 SMs, which is also what the plan assumes
    without a device)."""
    if torch.cuda.is_available() and torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the recorded sizes are for 148 SMs")
    desc = build_model(shape, CPU).descriptor()
    lib = L.load()
    L.set_precision(mode)
    got = [_sizes(lib, desc, b) for b in BATCHES]
    k = L.backward_kernels(desc)
    got.append((int(k["reads_tc"]), int(k["cnn_tc"])))
    assert got == [tuple(v) for v in EXPECTED[shape.name][mode]]


# (forward workspace, backward workspace, saved bytes) per batch of BATCHES, then (reads_tc, cnn_tc) of the backward
EXPECTED = {
    'max_corner': {
        'fp32': [(1266432, 101692416, 0), (1275392, 101708800, 0), (1598464, 102298880, 0), (34617856, 404209408, 0), (1686272, 102460416, 0), (0, 0)],
        'tf32x3': [(1266432, 510071552, 0), (1373696, 175458304, 16480768), (3466240, 592467776, 432880704), (2623232, 791433152, 329946816), (4045568, 2037499392, 1877745664), (1, 1)],
        'tf32': [(1266432, 510071552, 0), (1373696, 175458304, 0), (3466240, 592467776, 0), (2623232, 791433152, 0), (4045568, 2037499392, 0), (1, 1)],
    },
    'min_corner': {
        'fp32': [(478976, 19550720, 0), (481792, 19554816, 0), (583680, 19702528, 0), (8337408, 61812480, 0), (610816, 19742720, 0), (0, 0)],
        'tf32x3': [(478976, 385687808, 0), (580096, 40028672, 5005824), (2451456, 169280832, 134090816), (1495296, 176412608, 99123904), (2970112, 588948992, 553713664), (1, 1)],
        'tf32': [(478976, 385687808, 0), (580096, 40028672, 0), (2451456, 169280832, 0), (1495296, 176412608, 0), (2970112, 588948992, 0), (1, 1)],
    },
    'deep_odd': {
        'fp32': [(1753856, 108244480, 0), (1760512, 108256256, 0), (2000640, 108680192, 0), (22957056, 442259456, 0), (2065920, 108796416, 0), (0, 0)],
        'tf32x3': [(1753856, 566329600, 0), (1858816, 244946944, 30245376), (3868416, 1006434880, 791289920), (3367936, 1155540160, 606827200), (4425216, 3681235968, 3465969664), (1, 1)],
        'tf32': [(1753856, 566329600, 0), (1858816, 244946944, 0), (3868416, 1006434880, 0), (3367936, 1155540160, 0), (4425216, 3681235968, 0), (1, 1)],
    },
    'e1': {
        'fp32': [(1177344, 92863488, 0), (1185792, 92878848, 0), (1490432, 93432064, 0), (32567040, 375047168, 0), (1573376, 93583616, 0), (0, 0)],
        'tf32x3': [(1177344, 496327424, 0), (1284096, 161713152, 16480768), (3358208, 578685760, 432880704), (2526208, 757355712, 329946816), (3932672, 2023707392, 1877745664), (1, 1)],
        'tf32': [(1177344, 496327424, 0), (1284096, 161713152, 0), (3358208, 578685760, 0), (2526208, 757355712, 0), (3932672, 2023707392, 0), (1, 1)],
    },
    'simt_limits': {
        'fp32': [(1555200, 153343744, 0), (1566208, 153364224, 0), (1963008, 154101760, 0), (51739392, 577829376, 0), (2071040, 154303744, 0), (0, 0)],
        'tf32x3': [(1555200, 504129024, 0), (1664512, 154005248, 0), (3830784, 167150144, 0), (52525824, 583518912, 0), (4430336, 170689280, 0), (0, 1)],
        'tf32': [(1555200, 504129024, 0), (1664512, 154005248, 0), (3830784, 167150144, 0), (52525824, 583518912, 0), (4430336, 170689280, 0), (0, 1)],
    },
    'd_read_32': {
        'fp32': [(1459968, 125948928, 0), (1468416, 125964288, 0), (1773056, 126517504, 0), (33631232, 497216768, 0), (1856000, 126669056, 0), (0, 0)],
        'tf32x3': [(1459968, 476734208, 0), (1566720, 126605312, 0), (3640832, 139565888, 0), (34417664, 502906304, 0), (4215296, 143054592, 0), (0, 1)],
        'tf32': [(1459968, 476734208, 0), (1566720, 126605312, 0), (3640832, 139565888, 0), (34417664, 502906304, 0), (4215296, 143054592, 0), (0, 1)],
    },
    'd_info_seq_33': {
        'fp32': [(1477376, 126494976, 0), (1486592, 126511872, 0), (1818880, 127120384, 0), (34051328, 497786880, 0), (1909248, 127287040, 0), (0, 0)],
        'tf32x3': [(1477376, 477280256, 0), (1584896, 127152896, 0), (3686656, 140168768, 0), (34837760, 503476416, 0), (4268544, 143672576, 0), (0, 1)],
        'tf32': [(1477376, 477280256, 0), (1584896, 127152896, 0), (3686656, 140168768, 0), (34837760, 503476416, 0), (4268544, 143672576, 0), (0, 1)],
    },
    'h_12': {
        'fp32': [(1506048, 126250240, 0), (1514496, 126265600, 0), (1819136, 126818816, 0), (34458624, 497518080, 0), (1902080, 126970368, 0), (0, 0)],
        'tf32x3': [(1506048, 477035520, 0), (1612800, 126906624, 0), (3686912, 139867200, 0), (35245056, 503207616, 0), (4261376, 143355904, 0), (0, 1)],
        'tf32': [(1506048, 477035520, 0), (1612800, 126906624, 0), (3686912, 139867200, 0), (35245056, 503207616, 0), (4261376, 143355904, 0), (0, 1)],
    },
    'e_17': {
        'fp32': [(1443584, 122769920, 0), (1452032, 122785280, 0), (1756672, 123338496, 0), (32833280, 484972800, 0), (1839616, 123489792, 0), (0, 0)],
        'tf32x3': [(1443584, 473555200, 0), (1550336, 123426304, 0), (3624448, 136386880, 0), (33619712, 490662336, 0), (4198912, 139875328, 0), (0, 1)],
        'tf32': [(1443584, 473555200, 0), (1550336, 123426304, 0), (3624448, 136386880, 0), (33619712, 490662336, 0), (4198912, 139875328, 0), (0, 1)],
    },
    'k_7': {
        'fp32': [(1441536, 121729792, 0), (1449984, 121745152, 0), (1754624, 122298368, 0), (32831232, 481744640, 0), (1837568, 122449664, 0), (0, 0)],
        'tf32x3': [(1441536, 472515072, 0), (1548288, 122386176, 0), (3622400, 135346752, 0), (33617664, 487434176, 0), (4196864, 138835200, 0), (0, 1)],
        'tf32': [(1441536, 472515072, 0), (1548288, 122386176, 0), (3622400, 135346752, 0), (33617664, 487434176, 0), (4196864, 138835200, 0), (0, 1)],
    },
    'read_two_linears': {
        'fp32': [(1323776, 107150080, 0), (1332224, 107165440, 0), (1636864, 107718656, 0), (32713472, 420278784, 0), (1719808, 107870208, 0), (0, 0)],
        'tf32x3': [(1323776, 457935360, 0), (1430528, 107806464, 0), (3504640, 120767040, 0), (33499904, 425968320, 0), (4079104, 124255744, 0), (0, 1)],
        'tf32': [(1323776, 457935360, 0), (1430528, 107806464, 0), (3504640, 120767040, 0), (33499904, 425968320, 0), (4079104, 124255744, 0), (0, 1)],
    },
    'read_one_linear': {
        'fp32': [(1300224, 104239872, 0), (1308672, 104255232, 0), (1613312, 104808448, 0), (32689920, 407991296, 0), (1696256, 104960000, 0), (0, 0)],
        'tf32x3': [(1300224, 455025152, 0), (1406976, 104896256, 0), (3481088, 117856832, 0), (33476352, 413680832, 0), (4055552, 121345536, 0), (0, 1)],
        'tf32': [(1300224, 455025152, 0), (1406976, 104896256, 0), (3481088, 117856832, 0), (33476352, 413680832, 0), (4055552, 121345536, 0), (0, 1)],
    },
    'info_w32': {
        'fp32': [(1339136, 113206272, 0), (1350656, 113227776, 0), (1765888, 114002176, 0), (34339840, 445810688, 0), (1879040, 114214400, 0), (0, 0)],
        'tf32x3': [(1339136, 463991552, 0), (1448960, 113868800, 0), (3633664, 127050560, 0), (35126272, 451500224, 0), (4238336, 130599936, 0), (0, 1)],
        'tf32': [(1339136, 463991552, 0), (1448960, 113868800, 0), (3633664, 127050560, 0), (35126272, 451500224, 0), (4238336, 130599936, 0), (0, 1)],
    },
    'info_tile_gemm': {
        'fp32': [(1426176, 121532672, 0), (1434624, 121548032, 0), (1739264, 122101248, 0), (32815872, 481547520, 0), (1822208, 122252544, 0), (0, 0)],
        'tf32x3': [(1426176, 544788480, 0), (1532928, 213451008, 19888640), (3607040, 715751488, 521616448), (2775040, 952067520, 398497472), (4181504, 2465253120, 2270961664), (1, 1)],
        'tf32': [(1426176, 544788480, 0), (1532928, 213451008, 0), (3607040, 715751488, 0), (2775040, 952067520, 0), (4181504, 2465253120, 0), (1, 1)],
    },
    'n_info_9': {
        'fp32': [(1429248, 120957184, 0), (1437696, 120972544, 0), (1742336, 121525760, 0), (32818944, 480972288, 0), (1825280, 121677312, 0), (0, 0)],
        'tf32x3': [(1429248, 544212992, 0), (1536000, 212875520, 19888640), (3610112, 715176000, 521616448), (2778112, 951492288, 398497472), (4184576, 2464677888, 2270961664), (1, 1)],
        'tf32': [(1429248, 544212992, 0), (1536000, 212875520, 0), (3610112, 715176000, 0), (2778112, 951492288, 0), (4184576, 2464677888, 0), (1, 1)],
    },
    'n_info_128': {
        'fp32': [(1450752, 122387200, 0), (1459200, 122402560, 0), (1763840, 122955776, 0), (32840448, 482402304, 0), (1846784, 123107328, 0), (0, 0)],
        'tf32x3': [(1450752, 545643008, 0), (1557504, 214305536, 19888640), (3631616, 716606016, 521616448), (2799616, 952922304, 398497472), (4206080, 2466107904, 2270961664), (1, 1)],
        'tf32': [(1450752, 545643008, 0), (1557504, 214305536, 0), (3631616, 716606016, 0), (2799616, 952922304, 0), (4206080, 2466107904, 0), (1, 1)],
    },
    'hap_50': {
        'fp32': [(1199616, 121892608, 0), (1208064, 121907968, 0), (1512704, 122461184, 0), (32589312, 481907456, 0), (1595648, 122612480, 0), (0, 0)],
        'tf32x3': [(1199616, 194363136, 0), (1208064, 213169920, 0), (1512704, 703063040, 0), (1762048, 946737920, 0), (1595648, 2449227520, 0), (1, 0)],
        'tf32': [(1199616, 194363136, 0), (1208064, 213169920, 0), (1512704, 703063040, 0), (1762048, 946737920, 0), (1595648, 2449227520, 0), (1, 0)],
    },
    'hap_64': {
        'fp32': [(1199616, 122082048, 0), (1208064, 122097408, 0), (1512704, 122650624, 0), (32589312, 482096896, 0), (1595648, 122801920, 0), (0, 0)],
        'tf32x3': [(1199616, 194552576, 0), (1208064, 213359360, 0), (1512704, 703252480, 0), (1762048, 946927360, 0), (1595648, 2449416960, 0), (1, 0)],
        'tf32': [(1199616, 194552576, 0), (1208064, 213359360, 0), (1512704, 703252480, 0), (1762048, 946927360, 0), (1595648, 2449416960, 0), (1, 0)],
    },
}
