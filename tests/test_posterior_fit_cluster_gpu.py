"""The fused posterior fit pass on clusters of C = 1, 2, 4, 8 and 16 CTAs (pmt_posterior_fit_pass, _many): every output of
every width is bit for bit the one-CTA pass (PMT_POSTERIOR_CTAS=1), over golden and 300 k synthetic records, fp16 and fp32,
K = 1, 5, 16, the model configurations and batch sizes 1 ... 1000; the width the library chooses without the override;
and learn_priors_and_spectra / learn_priors_and_spectra_together at that width against the one-CTA runs."""
import copy
import functools

import pytest
import torch

from permutect_b200.engine import library as L
from test_posterior_fit_many_gpu import DEV, TAGS, Problem, _golden, _many, _mixed_problems, _model, _records, _single, _synthetic

pytestmark = pytest.mark.gpu
WIDTHS = (1, 2, 4, 8, 16)
KEYS = ("raw", "m", "v", "step", "losses", "tc", "snv", "ctx")


def _width(monkeypatch, ctas):
    """Forces the cluster width (None: the library's choice)."""
    if ctas is None:
        monkeypatch.delenv("PMT_POSTERIOR_CTAS", raising=False)
    else:
        monkeypatch.setenv("PMT_POSTERIOR_CTAS", str(ctas))


def _ctas(problems, bufs=None):
    bufs = bufs if bufs is not None else [p.buffers() for p in problems]
    return L.posterior_fit_ctas([p.struct(b) for p, b in zip(problems, bufs)])


@functools.lru_cache(maxsize=1)
def _synthetic_300k():
    return _synthetic(300_000)


def _case(name):
    z, ia, fa = _golden()
    if name.startswith("synthetic"):
        ia, fa = _synthetic_300k()
    return {
        "golden-default-b64": lambda: Problem(_model(z, "default"), _records(ia, fa, 64), 0.05, context=True),
        "golden-het_beta-fp16-b7": lambda: Problem(_model(z, "het_beta"), _records(ia, fa, 7, fp16=True), 0.05, context=False),
        "golden-no_germline-K1-b100": lambda: Problem(_model(z, "no_germline", n_components=1), _records(ia, fa, 100), 0.01, context=True),
        "golden-K16-fp16-b1000": lambda: Problem(_model(z, "default", 0.1, seed=2, n_components=16), _records(ia, fa, 1000, fp16=True), 0.05),
        "golden-40-records-b1": lambda: Problem(_model(z, "het_beta", 0.2, seed=3), _records(ia[:40], fa[:40], 1), 0.05, context=True),
        "golden-3-records-b64": lambda: Problem(_model(z, "no_germline"), _records(ia[:3], fa[:3], 64), 0.05, totals=False),
        "golden-70-records-b1000": lambda: Problem(_model(z, "default", 0.1, seed=5), _records(ia[:70], fa[:70], 1000), 0.05, context=True),
        "synthetic-default-fp16-b64": lambda: Problem(_model(z, "default", 0.1, seed=4), _records(ia, fa, 64, fp16=True), 0.001, context=True),
        "synthetic-het_beta-K16-b1000": lambda: Problem(_model(z, "het_beta", n_components=16), _records(ia, fa, 1000), 0.002, context=False),
        "synthetic-no_germline-K1-b100": lambda: Problem(_model(z, "no_germline", 0.1, seed=6, n_components=1), _records(ia, fa, 100),
                                                         0.002, context=True),
    }[name]()


CASES = ["golden-default-b64", "golden-het_beta-fp16-b7", "golden-no_germline-K1-b100", "golden-K16-fp16-b1000",
         "golden-40-records-b1", "golden-3-records-b64", "golden-70-records-b1000", "synthetic-default-fp16-b64",
         "synthetic-het_beta-K16-b1000", "synthetic-no_germline-K1-b100"]


def _three_passes(problem, run):
    """Every output after each of three passes that carry the spectra, Adam state and totals."""
    b = problem.buffers()
    seen = []
    for _ in range(3):
        run(b)
        seen.append({k: b[k].clone() for k in KEYS})
    return seen


def _assert_same(got, want, what):
    for i, (g, w) in enumerate(zip(got, want)):
        for k in KEYS:
            assert torch.equal(g[k], w[k]), f"{what}, pass {i}: {k} differs from the one-CTA pass"
        assert bool(torch.isfinite(g["losses"]).all()), f"{what}, pass {i}: non-finite batch loss"


@pytest.mark.parametrize("name", CASES)
def test_every_width_gives_the_one_cta_bits(monkeypatch, name):
    problem = _case(name)
    _width(monkeypatch, 1)
    assert _ctas([problem]) == 1
    want = _three_passes(problem, lambda b: _single(problem, b))
    assert int(want[-1]["step"]) == 3 * len(problem.records)
    for ctas in WIDTHS[1:]:
        _width(monkeypatch, ctas)
        assert _ctas([problem]) == ctas
        _assert_same(_three_passes(problem, lambda b: _single(problem, b)), want, f"{name}, C = {ctas}")


def _alone(problems):
    """Each problem's pass by pmt_posterior_fit_pass on one CTA."""
    bufs = [p.buffers() for p in problems]
    for p, b in zip(problems, bufs):
        _single(p, b)
    return bufs


def _assert_many(problems, got, want, ctas):
    for i, (p, g, w) in enumerate(zip(problems, got, want)):
        for k in KEYS:
            assert torch.equal(g[k], w[k]), f"C = {ctas}, problem {i} ({p.records.size()} records, batch {p.records.batch_size}): {k} differs"


@pytest.mark.parametrize("ctas", WIDTHS[1:])
def test_many_at_a_forced_width_is_each_problem_alone(monkeypatch, ctas):
    problems = _mixed_problems()
    _width(monkeypatch, 1)
    want = _alone(problems)
    _width(monkeypatch, ctas)
    assert _ctas(problems) == ctas
    got = [p.buffers() for p in problems]
    _many(problems, got)
    _assert_many(problems, got, want, ctas)


def _one_wave_limit(ctas):
    """The most problems whose clusters of `ctas` CTAs are resident at once, from the library's own choice: the largest n for
    which n problems of batch 1000 get a width of at least `ctas`."""
    z, ia, fa = _golden()
    p = Problem(_model(z, "default"), _records(ia, fa, 1000), 0.05)
    s = p.struct(p.buffers())
    n_sm = torch.cuda.get_device_properties(DEV).multi_processor_count
    limit = max(n for n in range(1, n_sm + 1) if L.posterior_fit_ctas([s] * n) >= ctas)
    assert all(L.posterior_fit_ctas([s] * n) >= ctas for n in range(1, limit + 1))
    return limit


@pytest.mark.parametrize("ctas", [4, 16])
def test_many_at_the_one_wave_limit_and_past_it(monkeypatch, ctas):
    _width(monkeypatch, None)
    limit = _one_wave_limit(ctas)
    z, ia, fa = _golden()
    for n in (limit, limit + 5):
        problems = []
        for i in range(n):
            lo, m = (11 * i) % (len(ia) - 120), 20 + (i * 37) % 100
            problems.append(Problem(_model(z, TAGS[i % 3], 0.05 * (i % 4), seed=i, n_components=(1, 5, 16)[i % 3]),
                                    _records(ia[lo:lo + m], fa[lo:lo + m], (64, 7, 100, 1000, 1)[i % 5], fp16=i % 2 == 1), 0.05,
                                    totals=i % 5 != 0, context=i % 3 == 0))
        _width(monkeypatch, 1)
        want = _alone(problems)
        _width(monkeypatch, ctas)
        assert _ctas(problems) == ctas
        got = [p.buffers() for p in problems]
        _many(problems, got)
        _assert_many(problems, got, want, ctas)


def test_the_chosen_width(monkeypatch):
    _width(monkeypatch, None)
    z, ia, fa = _golden()
    si, sf = _synthetic(20_000)
    n_sm = torch.cuda.get_device_properties(DEV).multi_processor_count

    def one(batch_size, n=len(si)):
        p = Problem(_model(z, "default"), _records(si[:n], sf[:n], batch_size), 0.05)
        return p.struct(p.buffers())

    assert L.posterior_fit_ctas([one(64)]) == 4          # a warp per record on four SMs
    assert L.posterior_fit_ctas([one(1000)]) == 16
    assert L.posterior_fit_ctas([one(256)]) == 16
    assert L.posterior_fit_ctas([one(100)]) == 4          # ceil(100 / 16) = 7
    assert L.posterior_fit_ctas([one(17)]) == 2
    assert L.posterior_fit_ctas([one(16)]) == 1
    assert L.posterior_fit_ctas([one(7)]) == 1
    assert L.posterior_fit_ctas([one(1000, n=40)]) == 2   # the batch is the 40 records there are
    # the widest batch decides, and every problem's cluster must be resident at once
    assert L.posterior_fit_ctas([one(7), one(64), one(1)]) == 4
    c16 = L.posterior_fit_ctas([one(1000)] * 16)
    assert c16 in (2, 4, 8) and 16 * c16 <= n_sm
    assert L.posterior_fit_ctas([one(1000)] * n_sm) == 1
    assert L.posterior_fit_ctas([one(1000)] * (n_sm + 3)) == 1
    # the override wins, whatever the problems
    for ctas in WIDTHS:
        _width(monkeypatch, ctas)
        assert L.posterior_fit_ctas([one(1)] * (n_sm + 3)) == ctas


def _learn(model, records, iterations=3):
    return model.learn_priors_and_spectra(records, num_iterations=iterations, ignored_to_non_ignored_ratio=10.0, learning_rate=0.05)


def _assert_models_equal(got, want):
    sg, sw = got.state_dict(), want.state_dict()
    assert sg.keys() == sw.keys()
    for k in sg:
        assert torch.equal(sg[k], sw[k]), f"{k} differs from the one-CTA run"


def test_learn_priors_and_spectra_at_the_chosen_width(monkeypatch):
    z, ia, fa = _golden()
    si, sf = _synthetic(20_000)
    for model, records in ((_model(z, "default"), _records(ia, fa, 64)), (_model(z, "het_beta", 0.1, seed=9), _records(si, sf, 100, fp16=True))):
        _width(monkeypatch, None)
        p = Problem(model, records, 0.05)
        assert _ctas([p]) == 4
        one_cta = copy.deepcopy(model)
        got = _learn(model, records)
        _width(monkeypatch, 1)
        assert _ctas([p]) == 1
        want = _learn(one_cta, records)
        assert got == want
        _assert_models_equal(model, one_cta)


def test_together_at_the_chosen_width(monkeypatch):
    from permutect_b200.architecture.posterior_model import learn_priors_and_spectra_together
    z, ia, fa = _golden()
    models = [_model(z, "default"), _model(z, "het_beta", 0.1, seed=7), _model(z, "no_germline"), _model(z, "default", 0.2, seed=8)]
    records = [_records(ia, fa, 16), _records(ia[:200], fa[:200], 64, fp16=True), _records(ia, fa, 7), _records(ia[10:], fa[10:], 300)]
    one_cta = [copy.deepcopy(m) for m in models]
    _width(monkeypatch, None)
    assert _ctas([Problem(m, r, 0.05) for m, r in zip(models, records)]) == 16
    got = learn_priors_and_spectra_together(models, records, 4, 10.0, learning_rate=0.05)
    _width(monkeypatch, 1)
    want = learn_priors_and_spectra_together(one_cta, records, 4, 10.0, learning_rate=0.05)
    assert got == want
    for m, w in zip(models, one_cta):
        _assert_models_equal(m, w)


def test_cluster_pass_is_reproducible(monkeypatch):
    problem = _case("synthetic-default-fp16-b64")
    _width(monkeypatch, None)
    assert _ctas([problem]) == 4
    first = _three_passes(problem, lambda b: _single(problem, b))
    _assert_same(_three_passes(problem, lambda b: _single(problem, b)), first, "second run")
    problems = _mixed_problems()
    _width(monkeypatch, 8)
    runs = []
    for _ in range(2):
        bufs = [p.buffers() for p in problems]
        _many(problems, bufs)
        runs.append(bufs)
    _assert_many(problems, runs[1], runs[0], 8)
