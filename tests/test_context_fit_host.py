"""CPU-only checks of the device context fit's C-ABI surface (pmt_snv_context_fit_many: exported, bound, sized, every bad
argument refused with its message before anything reaches a device) and of the ``context_fit`` argument of the posterior
model's two fitting entry points."""
import pytest
import torch

from permutect_b200.architecture import snv_context_priors as S
from permutect_b200.architecture.posterior_model import PosteriorModel, learn_priors_and_spectra_together
from permutect_b200.engine import library as L

FAKE = 256          # never dereferenced: every refusal below comes before anything is enqueued
ARGS = ("total_sc", "snv_sc", "elbo_draws", "mean_draws", "rates_out", "mu_out", "log_sigma_out", "n_iter_out",
        "func_evals_out", "workspace")
OPTIONAL = ("mu_out", "log_sigma_out", "n_iter_out", "func_evals_out")


def _call(n=3, null=None, workspace_bytes=None):
    lib = L.load()
    ptrs = {a: (None if a == null else FAKE) for a in ARGS}
    if workspace_bytes is None:
        workspace_bytes = lib.pmt_snv_context_fit_workspace_size(max(n, 1))
    rc = lib.pmt_snv_context_fit_many(n, *[ptrs[a] for a in ARGS], workspace_bytes, None)
    return rc, lib.pmt_last_error().decode()


def test_context_fit_symbols_are_exported_and_bound():
    lib = L.load()
    assert lib.pmt_abi_version() == L.PMT_ABI_VERSION == 4
    for name in ("pmt_snv_context_fit_many", "pmt_snv_context_fit_workspace_size"):
        assert name in L.EXPORTED_SYMBOLS
        assert getattr(lib, name).argtypes is not None


def test_workspace_size_is_linear_in_the_problem_count():
    lib = L.load()
    size = lib.pmt_snv_context_fit_workspace_size
    per_problem = size(2) - size(1)
    assert per_problem >= 2 * 100 * 388 * 8                       # the L-BFGS history of one problem
    for n in (1, 7, 148, 299, 1000):
        assert size(n) == size(1) + (n - 1) * per_problem
    assert size(0) == 0 and size(-1) == 0


@pytest.mark.parametrize("n", [0, -2])
def test_no_problems_is_refused(n):
    rc, msg = _call(n=n)
    assert rc != 0 and f"n {n} < 1" in msg


@pytest.mark.parametrize("null", [a for a in ARGS if a not in OPTIONAL])
def test_null_required_pointer_is_refused(null):
    rc, msg = _call(null=null)
    assert rc != 0 and f"null {null}" in msg


def test_short_workspace_is_refused():
    lib = L.load()
    need = lib.pmt_snv_context_fit_workspace_size(3)
    rc, msg = _call(workspace_bytes=need - 1)
    assert rc != 0 and "workspace too small" in msg and str(need) in msg


def test_draw_tables_are_the_host_fits_draws():
    elbo, mean = S.draw_tables("cpu")
    assert elbo.shape == (64, S.DIM) and mean.shape == (1000, S.DIM) and elbo.dtype == mean.dtype == torch.float64
    assert torch.equal(elbo, S._sobol_normal(64, S.DIM, seed=1234))
    assert torch.equal(mean, S._sobol_normal(1000, S.DIM, seed=4321))


def test_host_fit_parts_give_the_host_fit():
    g = torch.Generator().manual_seed(3)
    total = torch.full((12, 16), 1e6, dtype=torch.float64)
    snv = torch.round(total * 3e-6 * torch.rand(12, 16, dtype=torch.float64, generator=g))
    mu, log_sigma, n_iter, func_evals = S.fit_variational_sc(total, snv)
    assert mu.shape == log_sigma.shape == (S.DIM,)
    assert 0 < n_iter <= 300 and n_iter <= func_evals <= 375
    assert torch.equal(S.mean_rates_sc(mu, log_sigma, total, snv), S.fit_mutation_rates_sc(total, snv))


# neutral ids: an id "gpu" would put the test under the gpu marker's keyword
@pytest.mark.parametrize("value", ["gpu", "cpu", "", None, "Device"], ids=["value0", "value1", "value2", "value3", "value4"])
def test_unknown_context_fit_is_refused(value):
    model = PosteriorModel(-10.0, -10.0, device="cpu")
    with pytest.raises(ValueError, match="context_fit"):
        model.learn_priors_and_spectra([], 2, 0.5, context_fit=value)
    with pytest.raises(ValueError, match="context_fit"):
        learn_priors_and_spectra_together([model], [object()], 2, 0.5, context_fit=value)
