"""CPU-only checks of pmt_posterior_fit_pass's C-ABI surface: exported, bound, sized, and loud about bad arguments before
anything reaches a device."""
import ctypes as C

import pytest

from permutect_b200.engine import library as L


def test_fit_pass_symbols_are_exported_and_bound():
    lib = L.load()
    assert lib.pmt_abi_version() == L.PMT_ABI_VERSION == 4
    for name in ("pmt_posterior_fit_pass", "pmt_posterior_fit_pass_workspace_size"):
        assert name in L.EXPORTED_SYMBOLS
        assert getattr(lib, name).argtypes is not None


def test_fit_pass_workspace_size():
    lib = L.load()
    for k in (1, 5, 16):
        assert lib.pmt_posterior_fit_pass_workspace_size(k) > 0
    assert lib.pmt_posterior_fit_pass_workspace_size(17) == 0


def _call(lib, n_components=5, batch_size=64, workspace_bytes=None):
    desc = L.PmtPosteriorDesc(n_components, 16, 21, 0, 0, -1.0)
    if workspace_bytes is None:
        workspace_bytes = lib.pmt_posterior_fit_pass_workspace_size(5)
    fake = 256          # never dereferenced: every refusal below comes before the launch
    return lib.pmt_posterior_fit_pass(C.byref(desc), fake, fake, fake, fake, fake, 0.001, fake, 58, fake, L.F32, 16, 1000,
                                      batch_size, fake, None, None, None, fake, workspace_bytes, None)


@pytest.mark.parametrize("kwargs, message", [
    (dict(batch_size=0), "batch_size"),
    (dict(batch_size=-3), "batch_size"),
    (dict(n_components=17), "components"),
    (dict(n_components=0), "components"),
    (dict(workspace_bytes=16), "workspace too small"),
])
def test_fit_pass_refuses_bad_arguments(kwargs, message):
    lib = L.load()
    assert _call(lib, **kwargs) != 0
    assert message in lib.pmt_last_error().decode()


def test_posterior_records_refuse_an_empty_batch_size():
    from permutect_b200.architecture.posterior_model import PosteriorRecords
    with pytest.raises(ValueError, match="batch_size"):
        PosteriorRecords([[0] * 58], [[0.0] * 16], batch_size=0)
