"""CPU-only checks of pmt_posterior_fit_ctas (the cluster width of the fused posterior fit passes): exported and bound,
every bad argument refused with its problem's index, and a PMT_POSTERIOR_CTAS override outside the five widths refused by
the query and by both fit passes before anything reaches a device."""
import ctypes as C

import pytest

from permutect_b200.engine import library as L

FAKE = 256          # never dereferenced: every refusal below comes before anything is enqueued


def _problem(n_components=5, batch_size=64, n_records=1000):
    return L.PmtPosteriorFitProblem(L.PmtPosteriorDesc(n_components, 16, 21, 0, 0, -1.0), FAKE, FAKE, FAKE, FAKE, FAKE, 0.001,
                                    FAKE, 58, FAKE, L.F32, 16, n_records, batch_size, FAKE, None, None, None)


def _query(problems, n_problems=None):
    lib = L.load()
    arr = (L.PmtPosteriorFitProblem * max(len(problems), 1))(*problems)
    ctas = lib.pmt_posterior_fit_ctas(arr, len(problems) if n_problems is None else n_problems)
    return ctas, lib.pmt_last_error().decode()


def test_fit_ctas_is_exported_and_bound():
    lib = L.load()
    assert "pmt_posterior_fit_ctas" in L.EXPORTED_SYMBOLS
    assert lib.pmt_posterior_fit_ctas.argtypes is not None and lib.pmt_posterior_fit_ctas.restype is C.c_int


def test_null_problems_are_refused():
    lib = L.load()
    assert lib.pmt_posterior_fit_ctas(None, 3) == 0
    assert "pmt_posterior_fit_ctas: null argument" in lib.pmt_last_error().decode()


@pytest.mark.parametrize("n", [0, -2])
def test_no_problems_are_refused(n):
    ctas, msg = _query([_problem()], n_problems=n)
    assert ctas == 0 and "n_problems" in msg


@pytest.mark.parametrize("k", [0, 17])
def test_bad_components_are_refused_with_the_problem_index(k):
    ctas, msg = _query([_problem(), _problem(), _problem(n_components=k), _problem()])
    assert ctas == 0
    assert "problem 2" in msg and "components" in msg


def test_bad_problem_fields_are_refused_with_the_problem_index():
    bad = _problem()
    bad.params = None
    ctas, msg = _query([_problem(), bad])
    assert ctas == 0 and "problem 1" in msg and "null" in msg
    ctas, msg = _query([_problem(batch_size=0)])
    assert ctas == 0 and "problem 0" in msg and "batch_size" in msg


def _fit_pass(p):
    lib = L.load()
    return lib.pmt_posterior_fit_pass(C.byref(p.desc), p.params, p.raw_params, p.adam_m, p.adam_v, p.adam_step, p.learning_rate,
                                      p.int_array, p.int_stride, p.float_array, p.float_kind, p.float_stride, p.n_records,
                                      p.batch_size, p.batch_losses_out, None, None, None, FAKE,
                                      lib.pmt_posterior_fit_pass_workspace_size(5), None)


def _fit_pass_many(problems):
    lib = L.load()
    arr = (L.PmtPosteriorFitProblem * len(problems))(*problems)
    return lib.pmt_posterior_fit_pass_many(arr, len(problems), FAKE, lib.pmt_posterior_fit_pass_many_workspace_size(len(problems), 16),
                                           None)


@pytest.mark.parametrize("value", ["0", "3", "32", "-4", "abc", "4x", ""])
def test_override_outside_the_widths_is_refused(monkeypatch, value):
    monkeypatch.setenv("PMT_POSTERIOR_CTAS", value)
    lib = L.load()
    ctas, msg = _query([_problem()])
    assert ctas == 0 and "PMT_POSTERIOR_CTAS" in msg
    assert _fit_pass(_problem()) != 0
    assert "pmt_posterior_fit_pass: PMT_POSTERIOR_CTAS must be 1, 2, 4, 8 or 16" in lib.pmt_last_error().decode()
    assert _fit_pass_many([_problem(), _problem(n_components=16)]) != 0
    assert "pmt_posterior_fit_pass_many: PMT_POSTERIOR_CTAS" in lib.pmt_last_error().decode()


def test_python_query_raises_on_a_refusal():
    with pytest.raises(RuntimeError, match="problem 0.*components"):
        L.posterior_fit_ctas([_problem(n_components=0)])
