"""The device context fit (pmt_snv_context_fit_many, architecture/snv_context_priors.fit_context_models_on_device) against
the host fit (fit_mutation_rates_sc): the same method, so the same optimum to rounding, on converging inputs and on inputs
that run to max_iter; the model's own limits; launch independence; and the posterior model's fits with
context_fit="device" against "host"."""
import copy
import importlib.util
import os

import numpy as np
import pytest
import torch

from permutect_b200.architecture import snv_context_priors as S

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "posterior_model.npz")
pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _counts(seed, lo, hi, max_snv, empty=0.0):
    """Cell totals log-uniform in [10^lo, 10^hi], SNV counts up to max_snv, a fraction `empty` of cells with neither."""
    g = torch.Generator().manual_seed(seed)
    total = torch.round(10 ** (lo + (hi - lo) * torch.rand(12, 16, dtype=torch.float64, generator=g)))
    snv = torch.round(max_snv * torch.rand(12, 16, dtype=torch.float64, generator=g) ** 2)
    if empty:
        e = torch.rand(12, 16, generator=g) < empty
        total[e] = 0
        snv[e] = 0
    return total, snv


# (lo, hi, max SNVs, empty fraction) by seed % 5: the realistic ranges, sparse counts, no SNVs at all, empty cells
SHAPES = [(5, 8, 50, 0.0), (5, 6, 10, 0.0), (7, 8, 50, 0.1), (5, 8, 0, 0.0), (6, 7, 50, 0.3)]
CONVERGING_SEEDS = [s for s in range(1, 22)]


def _converging(seed):
    return _counts(seed, *SHAPES[seed % 5])


def _max_iter_case():
    """Totals near 1e7 with up to 300 SNVs per cell: the host fit stops at max_iter = 300."""
    g = torch.Generator().manual_seed(100)
    total = torch.round(1e7 * (1 + 0.2 * torch.rand(12, 16, dtype=torch.float64, generator=g)))
    snv = torch.round(300 * torch.rand(12, 16, dtype=torch.float64, generator=g))
    return total, snv


def _objective(mu, log_sigma, total, snv):
    """The host's objective -(mean_d lp(mu + exp(log_sigma) eps_d) + sum log_sigma), float64 on the CPU."""
    total, snv = S._clamped_inputs(total, snv)
    eps = S._sobol_normal(64, S.DIM, seed=1234)
    mu, log_sigma = mu.double().cpu(), log_sigma.double().cpu()
    lp, _ = S._log_joint(mu + torch.exp(log_sigma) * eps, total, snv)
    return float(-(lp.mean() + log_sigma.sum()))


def _device(cases):
    total = torch.stack([t for t, _ in cases]).to(DEV)
    snv = torch.stack([s for _, s in cases]).to(DEV)
    out = S.fit_context_models_on_device(total, snv, DEV)
    torch.cuda.synchronize()
    return [t.cpu() for t in out]


@pytest.fixture(scope="module")
def converging():
    """The host fits that stop well before max_iter, and the device fits of the same inputs in one launch."""
    cases, host = [], []
    for seed in CONVERGING_SEEDS:
        total, snv = _converging(seed)
        fit = S.fit_variational_sc(total, snv)
        if fit[2] < 250:
            cases.append((total, snv))
            host.append(fit)
        if len(cases) == 20:
            break
    assert len(cases) >= 18
    return cases, host, _device(cases)


def test_converging_inputs_reach_the_host_optimum(converging):
    """The objective is the primary check: the device optimum is never worse than the host's.  The rates of a flat optimum
    (most of all along empty cells) move with rounding: the host fit's own rates move by up to 8e-7, and its iteration
    count by 2, when only its draws change by one ulp, and every sum of the device fit runs in another order.  Where the
    optimum is flat the last iterations change the objective by nothing measurable, so the two fits stop some iterations
    apart (measured on a B200: up to 21 of the host's 193, the device objective 1.8e-14 from the host's at most).  The gaps
    are all measured and printed first, then held to 1e-4 (rates) and max(5, 20 %) (iterations)."""
    cases, host, (rates, mu, log_sigma, n_iter, func_evals) = converging
    obj, rate_gap, iter_gap = [], [], []
    for i, ((total, snv), (h_mu, h_ls, h_iter, h_evals)) in enumerate(zip(cases, host)):
        h_rates = S.mean_rates_sc(h_mu, h_ls, total, snv)
        f_dev, f_host = _objective(mu[i], log_sigma[i], total, snv), _objective(h_mu, h_ls, total, snv)
        obj.append((f_dev - f_host) / abs(f_host))
        rate_gap.append(float(((rates[i] - h_rates).abs() / h_rates.abs()).max()))
        iter_gap.append((int(n_iter[i]) - h_iter, h_iter))
        assert int(n_iter[i]) < 300 and int(n_iter[i]) <= int(func_evals[i]) <= 375
        # the device's rates are the mean over the mean draws at its own (mu, log_sigma)
        again = S.mean_rates_sc(mu[i], log_sigma[i], total, snv)
        np.testing.assert_allclose(rates[i].numpy(), again.numpy(), rtol=1e-12, atol=0)
    print(f"\n{len(cases)} converging inputs: relative rate gaps {[f'{g:.1e}' for g in sorted(rate_gap)]}; "
          f"max relative objective excess {max(obj):.2e}; n_iter gaps (device - host, host) {iter_gap}")
    assert max(obj) <= 1e-9
    assert max(rate_gap) < 1e-4
    assert all(abs(d) <= max(5, h // 5) for d, h in iter_gap)


def test_inputs_that_hit_max_iter():
    total, snv = _max_iter_case()
    h_mu, h_ls, h_iter, _ = S.fit_variational_sc(total, snv)
    rates, mu, log_sigma, n_iter, func_evals = _device([(total, snv)])
    assert h_iter == 300 and int(n_iter[0]) == 300
    f_dev, f_host = _objective(mu[0], log_sigma[0], total, snv), _objective(h_mu, h_ls, total, snv)
    gap = abs(f_dev - f_host) / abs(f_host)
    print(f"\nmax_iter input: relative objective gap {gap:.2e} (device {f_dev:.12g}, host {f_host:.12g})")
    assert gap < 1e-6


def _limits_counts(total_per_cell, seed=0):
    g = torch.Generator().manual_seed(seed)          # tests/test_snv_context_priors.py's counts
    true = 3e-6 * torch.exp(0.7 * torch.randn(12, 16, dtype=torch.float64, generator=g))
    total = torch.full((12, 16), float(total_per_cell), dtype=torch.float64)
    snv = torch.round(total * true + torch.sqrt(total * true) * torch.randn(12, 16, dtype=torch.float64, generator=g)).clamp(min=0)
    return true, total, snv


def _device_rates(total, snv):
    return S.fit_mutation_rates_sc_on_device([(total, snv)], DEV)[0]


def test_large_counts_give_the_empirical_rates():
    """Both fits run to max_iter on these counts, so where each stops is a point of an unconverged L-BFGS path: measured on
    a B200, the host's rates are within 0.16 % of snv / total and the device's within 2.3 %, at objectives 6e-8 apart
    (relative).  Hence 5 % here, where the host test has 2 %, and the max_iter criterion on the objective."""
    _, total, snv = _limits_counts(5e9)
    rates, mu, log_sigma, n_iter, _ = _device([(total, snv)])
    assert rates[0].shape == (12, 16) and rates.dtype == torch.float64
    np.testing.assert_allclose(rates[0].numpy(), (snv / total).numpy(), rtol=0.05)
    h_mu, h_ls, h_iter, _ = S.fit_variational_sc(total, snv)
    f_dev, f_host = _objective(mu[0], log_sigma[0], total, snv), _objective(h_mu, h_ls, total, snv)
    print(f"\nlarge counts: n_iter device {int(n_iter[0])} host {h_iter}, relative objective gap {abs(f_dev - f_host) / abs(f_host):.2e}")
    assert abs(f_dev - f_host) <= 1e-6 * abs(f_host)


def test_fit_is_deterministic_and_shrinks_empty_cells():
    true, total, snv = _limits_counts(2e7)
    total[3, 5], snv[3, 5] = 1000.0, 0.0
    a, b = _device_rates(total, snv), _device_rates(total, snv)
    assert torch.equal(a, b)
    assert torch.all(a > 0) and torch.all(torch.isfinite(torch.log(a)))
    row_mean = float((snv[3].sum() / total[3].sum()))
    assert 0.2 * row_mean < float(a[3, 5]) < 5 * row_mean
    _, total_s, snv_s = _limits_counts(2e5, seed=1)
    r = _device_rates(total_s, snv_s)
    assert 0.5 < float(r.mean() / true.mean()) < 2.0


def test_each_problem_is_independent_of_its_launch():
    distinct = [_converging(seed) for seed in range(1, 12)] + [_max_iter_case()]
    alone = [_device([c]) for c in distinct]
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    for n in (1, 7, sms, 2 * sms + 3):
        order = [(7 * i + n) % len(distinct) for i in range(n)]
        got = _device([distinct[k] for k in order])
        again = _device([distinct[k] for k in order])
        for a, b in zip(got, again):
            assert torch.equal(a, b), n
        for i, k in enumerate(order):
            for out, ref in zip(got, alone[k]):
                assert torch.equal(out[i], ref[0]), (n, i, k)


# ---- the posterior model's fits ------------------------------------------------------------------------------------

def _golden():
    z = np.load(GOLDEN)
    keep = z["int_array"][:, 5] <= 400
    return z, z["int_array"][keep], z["float_array"][keep]


def _model(z, tag, perturb=0.0, seed=0, n_components=None):
    from permutect_b200.architecture.posterior_model import PosteriorModel, SomaticSpectrum
    sd = {k[len(tag) + 4:]: z[k] for k in z.files if k.startswith(tag + "/sd/")}
    cfg = z[tag + "/cfg"]
    model = PosteriorModel(-3.0, -4.0, no_germline_mode=bool(cfg[0]), device=DEV, het_beta=None if cfg[1] < 0 else float(cfg[1]))
    model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
    if n_components is not None:
        model.spectra.somatic_spectrum = SomaticSpectrum(n_components).to(DEV)
    if perturb:
        g = torch.Generator().manual_seed(seed)
        with torch.no_grad():
            for t in model._raw_spectra_tensors():
                t.add_(perturb * torch.randn(t.shape, generator=g).to(DEV))
    return model


def _synthetic(n):
    spec = importlib.util.spec_from_file_location("time_posterior_fit", os.path.join(os.path.dirname(HERE), "profiles", "time_posterior_fit.py"))
    tpf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tpf)
    return tpf.synthetic_records(n, DEV)


def _check_device_against_host(model, loader, iterations, ratio, lr):
    host, dev = copy.deepcopy(model), copy.deepcopy(model)
    h = host.learn_priors_and_spectra(loader, iterations, ratio, learning_rate=lr, context_fit="host")
    d = dev.learn_priors_and_spectra(loader, iterations, ratio, learning_rate=lr, context_fit="device")
    first = iterations // 2 + 1        # every pass up to the first context fit's iteration runs on the same parameters
    assert h[:first] == d[:first]
    hist_gap = max(abs(a - b) / abs(a) for a, b in zip(h, d))
    ph = host.priors.somatic_snv_log_priors_rrra.detach().cpu()
    pd = dev.priors.somatic_snv_log_priors_rrra.detach().cpu()
    prior_gap = float((ph - pd).abs().max())
    print(f"\nhistories: max relative gap {hist_gap:.2e}; somatic_snv_log_priors_rrra: max |gap| {prior_gap:.2e}")
    assert hist_gap < 1e-5
    assert prior_gap < 1e-4
    assert float(pd[0:4, 0:4, 0:4, 0:4].std()) > 0


def test_learn_on_golden_records_device_against_host():
    from permutect_b200.architecture.posterior_model import PosteriorBatch
    z, ia, fa = _golden()
    loader = [PosteriorBatch(ia[s:s + 64], fa[s:s + 64], DEV) for s in range(0, len(ia), 64)]     # the batch-loader path
    _check_device_against_host(_model(z, "default"), loader, 6, 10.0, 0.05)


def test_learn_on_synthetic_records_device_against_host():
    from permutect_b200.architecture.posterior_model import PosteriorRecords
    z, _, _ = _golden()
    it, ft = _synthetic(100_000)
    _check_device_against_host(_model(z, "default"), PosteriorRecords(it, ft, batch_size=64, device=DEV), 6, 10.0, 0.001)


def test_together_on_device_matches_each_model_alone():
    from permutect_b200.architecture.posterior_model import PosteriorRecords, learn_priors_and_spectra_together
    z, ia, fa = _golden()
    models = [_model(z, "default"), _model(z, "het_beta", 0.1, seed=7, n_components=3), _model(z, "no_germline"),
              _model(z, "default", 0.2, seed=8, n_components=9)]
    fa = torch.as_tensor(fa)
    records = [PosteriorRecords(ia, fa.float(), 16, DEV), PosteriorRecords(ia[:200], fa[:200].half(), 64, DEV),
               PosteriorRecords(ia, fa.float(), 7, DEV), PosteriorRecords(ia[10:], fa[10:].float(), 300, DEV)]
    ratios, rates = [10.0, 5.0, 10.0, 20.0], [0.05, 0.05, 0.01, 0.05]
    alone = [copy.deepcopy(m) for m in models]
    want = [m.learn_priors_and_spectra(r, num_iterations=6, ignored_to_non_ignored_ratio=q, learning_rate=lr, context_fit="device")
            for m, r, q, lr in zip(alone, records, ratios, rates)]
    got = learn_priors_and_spectra_together(models, records, 6, ratios, learning_rate=rates, context_fit="device")
    assert got == want
    for i, (m, a) in enumerate(zip(models, alone)):
        sd, sa = m.state_dict(), a.state_dict()
        assert sd.keys() == sa.keys()
        for k in sd:
            assert torch.equal(sd[k], sa[k]), f"model {i}: {k} differs"
        assert float(m.priors.somatic_snv_log_priors_rrra.detach()[0:4, 0:4, 0:4, 0:4].std()) > 0
