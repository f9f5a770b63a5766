"""CPU-only checks of pmt_posterior_fit_pass_many's C-ABI surface (exported, bound, sized, every bad argument refused with
its problem's index before anything reaches a device), of learn_priors_and_spectra_together's argument checks, and of the
pool that runs the context fits of many models: bit for bit the in-process fits."""
import ctypes as C

import pytest
import torch

from permutect_b200.engine import library as L

FAKE = 256          # never dereferenced: every refusal below comes before anything is enqueued


def test_fit_pass_many_symbols_are_exported_and_bound():
    lib = L.load()
    assert lib.pmt_abi_version() == L.PMT_ABI_VERSION == 4
    for name in ("pmt_posterior_fit_pass_many", "pmt_posterior_fit_pass_many_workspace_size"):
        assert name in L.EXPORTED_SYMBOLS
        assert getattr(lib, name).argtypes is not None


def test_fit_pass_many_workspace_size():
    lib = L.load()
    for k in range(1, 17):
        assert lib.pmt_posterior_fit_pass_many_workspace_size(1, k) > 0
        assert lib.pmt_posterior_fit_pass_many_workspace_size(300, k) > 0
    for k in (0, 17, -1):
        assert lib.pmt_posterior_fit_pass_many_workspace_size(4, k) == 0
    assert lib.pmt_posterior_fit_pass_many_workspace_size(0, 5) == 0
    # the table and the context scratch grow with the problem count
    assert lib.pmt_posterior_fit_pass_many_workspace_size(8, 5) > lib.pmt_posterior_fit_pass_many_workspace_size(4, 5)


def _problem(n_components=5, batch_size=64, n_records=1000, null=None):
    p = L.PmtPosteriorFitProblem(L.PmtPosteriorDesc(n_components, 16, 21, 0, 0, -1.0), FAKE, FAKE, FAKE, FAKE, FAKE, 0.001,
                                 FAKE, 58, FAKE, L.F32, 16, n_records, batch_size, FAKE, None, None, None)
    if null is not None:
        setattr(p, null, None)
    return p


def _call(problems, workspace_bytes=None, n_problems=None):
    lib = L.load()
    n = len(problems) if n_problems is None else n_problems
    arr = (L.PmtPosteriorFitProblem * max(len(problems), 1))(*problems)
    if workspace_bytes is None:
        workspace_bytes = lib.pmt_posterior_fit_pass_many_workspace_size(max(n, 1), 16)
    rc = lib.pmt_posterior_fit_pass_many(arr, n, FAKE, workspace_bytes, None)
    return rc, lib.pmt_last_error().decode()


@pytest.mark.parametrize("null", ["params", "raw_params", "adam_m", "adam_v", "adam_step", "int_array", "float_array",
                                  "batch_losses_out"])
def test_null_pointer_in_problem_3_of_5_is_refused(null):
    rc, msg = _call([_problem() for _ in range(3)] + [_problem(null=null), _problem()])
    assert rc != 0
    assert "problem 3" in msg and "null" in msg


@pytest.mark.parametrize("kwargs, message", [
    (dict(n_components=17), "components"),
    (dict(n_components=0), "components"),
    (dict(batch_size=0), "batch_size"),
    (dict(batch_size=-3), "batch_size"),
    (dict(n_records=0), "no records"),
    (dict(n_records=(1 << 31) * 2, batch_size=1), "int32"),
])
def test_bad_problem_is_refused_with_its_index(kwargs, message):
    rc, msg = _call([_problem(), _problem(**kwargs), _problem()])
    assert rc != 0
    assert "problem 1" in msg and message in msg


def test_context_totals_need_haplotypes():
    bad = _problem()
    bad.desc.hap_len = 2
    bad.somatic_snv_totals_rrra = FAKE
    rc, msg = _call([_problem(), _problem(), bad])
    assert rc != 0 and "problem 2" in msg and "haplotypes" in msg


def test_no_problems_is_refused():
    rc, msg = _call([_problem()], n_problems=0)
    assert rc != 0 and "n_problems" in msg


def test_workspace_one_byte_short_is_refused():
    lib = L.load()
    problems = [_problem(n_components=k) for k in (1, 16, 5)]
    need = lib.pmt_posterior_fit_pass_many_workspace_size(3, 16)
    rc, msg = _call(problems, workspace_bytes=need - 1)
    assert rc != 0 and "workspace too small" in msg


def test_together_refuses_bad_lists():
    from permutect_b200.architecture.posterior_model import PosteriorModel, learn_priors_and_spectra_together
    with pytest.raises(ValueError, match="no models"):
        learn_priors_and_spectra_together([], [], 2, 10.0)
    model = PosteriorModel(-10.0, -10.0, device="cpu")
    with pytest.raises(ValueError, match="1 models but 2"):
        learn_priors_and_spectra_together([model], [None, None], 2, 10.0)
    with pytest.raises(ValueError, match="learning_rate"):
        learn_priors_and_spectra_together([model], [None], 2, 10.0, learning_rate=[0.1, 0.2])
    with pytest.raises(TypeError, match="PosteriorRecords"):
        learn_priors_and_spectra_together([model], [object()], 2, 10.0)


def test_context_fit_pool_gives_the_in_process_bits():
    from permutect_b200.architecture.snv_context_priors import ContextFitPool, fit_mutation_rates_sc
    g = torch.Generator().manual_seed(3)
    inputs = [(torch.round(torch.rand(12, 16, generator=g, dtype=torch.float64) * 5000 + 100),
               torch.round(torch.rand(12, 16, generator=g, dtype=torch.float64) * 40)) for _ in range(5)]
    pool = ContextFitPool(2)
    try:
        got = pool.map(inputs)
    finally:
        pool.close()
    want = [fit_mutation_rates_sc(*x) for x in inputs]
    assert all(torch.equal(a, b) for a, b in zip(got, want))
