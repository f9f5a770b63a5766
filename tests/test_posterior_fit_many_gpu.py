"""pmt_posterior_fit_pass_many (the fit passes of many samples' posterior models, a CTA each, in one launch) against
pmt_posterior_fit_pass run on each problem alone, bit for bit: one pass, carried Adam state, more problems than SMs, mixed
K; and learn_priors_and_spectra_together against each model's own learn_priors_and_spectra."""
import copy
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "posterior_model.npz")
pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TAGS = ("default", "het_beta", "no_germline")


def _golden():
    z = np.load(GOLDEN)
    keep = z["int_array"][:, 5] <= 400         # rows whose fp32 lgamma rounding stays small (test_posterior_model.py)
    return z, z["int_array"][keep], z["float_array"][keep]


def _model(z, tag, perturb=0.0, seed=0, n_components=None):
    from permutect_b200.architecture.posterior_model import PosteriorModel, SomaticSpectrum
    sd = {k[len(tag) + 4:]: z[k] for k in z.files if k.startswith(tag + "/sd/")}
    cfg = z[tag + "/cfg"]
    model = PosteriorModel(-3.0, -4.0, no_germline_mode=bool(cfg[0]), device=DEV, het_beta=None if cfg[1] < 0 else float(cfg[1]))
    model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
    model.priors.use_context_dependent_snv_priors = bool(cfg[2])
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


def _records(ia, fa, batch_size, fp16=False):
    from permutect_b200.architecture.posterior_model import PosteriorRecords
    fa = torch.as_tensor(fa)
    return PosteriorRecords(ia, fa.half() if fp16 else fa.float(), batch_size=batch_size, device=DEV)


class Problem:
    """A model's arguments of one pass (constant) and the buffers one run of it writes (fresh per run)."""

    def __init__(self, model, records, lr, totals=True, context=None):
        if context is not None:
            model.priors.use_context_dependent_snv_priors = context
        self.model, self.records, self.lr, self.totals = model, records, lr, totals
        self.it, self.ft, self.desc, self.flat = model._inputs(records)

    def buffers(self):
        raw = torch.cat([t.detach().reshape(-1) for t in self.model._raw_spectra_tensors()]).float().contiguous()
        return {"raw": raw, "m": torch.zeros_like(raw), "v": torch.zeros_like(raw), "step": torch.zeros(1, dtype=torch.int64, device=DEV),
                "losses": torch.full((len(self.records),), float("nan"), device=DEV), "tc": torch.zeros((5, 5), device=DEV),
                "snv": torch.zeros((5, 5, 5, 5), device=DEV), "ctx": torch.zeros((5, 5, 5, 5), device=DEV)}

    def struct(self, b):
        from permutect_b200.engine import library as L
        tot = (lambda k: b[k].data_ptr()) if self.totals else (lambda k: None)
        return L.PmtPosteriorFitProblem(self.desc, self.flat.data_ptr(), b["raw"].data_ptr(), b["m"].data_ptr(), b["v"].data_ptr(),
                                        b["step"].data_ptr(), self.lr, self.it.data_ptr(), self.it.stride(0), self.ft.data_ptr(),
                                        L.F16 if self.ft.dtype == torch.float16 else L.F32, self.ft.stride(0), self.records.size(),
                                        self.records.batch_size, b["losses"].data_ptr(), tot("tc"), tot("snv"), tot("ctx"))


def _single(problem, b):
    """One pmt_posterior_fit_pass of `problem` on its buffers `b`."""
    from permutect_b200.engine import library as L
    lib = L.load()
    s = problem.struct(b)
    ws = torch.empty(int(lib.pmt_posterior_fit_pass_workspace_size(s.desc.n_components)), dtype=torch.uint8, device=DEV)
    L.check(lib.pmt_posterior_fit_pass(C.byref(s.desc), s.params, s.raw_params, s.adam_m, s.adam_v, s.adam_step, s.learning_rate,
                                       s.int_array, s.int_stride, s.float_array, s.float_kind, s.float_stride, s.n_records, s.batch_size,
                                       s.batch_losses_out, s.posterior_totals_tc, s.somatic_snv_totals_rrra, s.snv_context_totals_rrra,
                                       ws.data_ptr(), ws.numel(), torch.cuda.current_stream(DEV).cuda_stream))
    torch.cuda.synchronize(DEV)


def _many(problems, bufs):
    """One pmt_posterior_fit_pass_many of all `problems`, problem i on its buffers bufs[i]."""
    from permutect_b200.engine import library as L
    lib = L.load()
    n = len(problems)
    arr = (L.PmtPosteriorFitProblem * n)(*[p.struct(b) for p, b in zip(problems, bufs)])
    max_k = max(p.desc.n_components for p in problems)
    ws = torch.empty(int(lib.pmt_posterior_fit_pass_many_workspace_size(n, max_k)), dtype=torch.uint8, device=DEV)
    L.check(lib.pmt_posterior_fit_pass_many(arr, n, ws.data_ptr(), ws.numel(), torch.cuda.current_stream(DEV).cuda_stream))
    torch.cuda.synchronize(DEV)


def _assert_bitwise(problems, got, want):
    for i, (p, g, w) in enumerate(zip(problems, got, want)):
        for k in w:
            assert torch.equal(g[k], w[k]), f"problem {i} ({p.records.size()} records, batch {p.records.batch_size}): {k} differs"
        assert bool(torch.isfinite(g["losses"]).all()), f"problem {i}: non-finite batch loss"


def _mixed_problems():
    """Eight problems: the golden configurations and perturbed copies; 1, 63, 64, 65, the golden set and thousands of
    records; batch sizes 1, 16, 64, 100 and larger than the record count; fp16 and fp32; totals and context priors on
    for some."""
    z, ia, fa = _golden()
    si, sf = _synthetic(5000)
    return [
        Problem(_model(z, "default"), _records(ia[:1], fa[:1], 64), 0.05),
        Problem(_model(z, "het_beta"), _records(ia[:63], fa[:63], 64, fp16=True), 0.05, totals=False),
        Problem(_model(z, "no_germline"), _records(ia[:64], fa[:64], 1), 0.01, context=True),
        Problem(_model(z, "default", 0.2, seed=1), _records(ia[:65], fa[:65], 64), 0.05, context=True),
        Problem(_model(z, "het_beta", 0.2, seed=2), _records(si, sf, 64, fp16=True), 0.001, context=True),
        Problem(_model(z, "no_germline", 0.2, seed=3), _records(si[:3000], sf[:3000], 100), 0.002, totals=False),
        Problem(_model(z, "default", 0.1, seed=4), _records(ia, fa, 16, fp16=True), 0.05),
        Problem(_model(z, "het_beta", 0.1, seed=5), _records(ia[5:105], fa[5:105], 1000), 0.05, context=False),
    ]


def test_one_pass_is_bitwise_each_problem_alone():
    problems = _mixed_problems()
    want = [p.buffers() for p in problems]
    for p, b in zip(problems, want):
        _single(p, b)
    got = [p.buffers() for p in problems]
    _many(problems, got)
    _assert_bitwise(problems, got, want)
    assert [int(b["step"]) for b in got] == [len(p.records) for p in problems]


def test_carried_state_over_three_passes_is_bitwise():
    problems = _mixed_problems()
    want = [p.buffers() for p in problems]
    got = [p.buffers() for p in problems]
    for _ in range(3):
        for p, b in zip(problems, want):
            _single(p, b)
        _many(problems, got)
    _assert_bitwise(problems, got, want)
    assert [int(b["step"]) for b in got] == [3 * len(p.records) for p in problems]


def test_more_problems_than_sms():
    n_sm = torch.cuda.get_device_properties(DEV).multi_processor_count
    z, ia, fa = _golden()
    problems = []
    for i in range(2 * n_sm + 7):
        lo = (7 * i) % (len(ia) - 40)
        n = 1 + (i * 13) % 40
        problems.append(Problem(_model(z, TAGS[i % 3], 0.05 * (i % 4), seed=i), _records(ia[lo:lo + n], fa[lo:lo + n], 1 + i % 9, fp16=i % 2 == 1),
                                0.05, totals=i % 5 != 0, context=i % 3 == 0))
    want = [p.buffers() for p in problems]
    for p, b in zip(problems, want):
        _single(p, b)
    got = [p.buffers() for p in problems]
    _many(problems, got)
    _assert_bitwise(problems, got, want)


def test_mixed_components_in_one_launch():
    z, ia, fa = _golden()
    problems = [Problem(_model(z, TAGS[i % 3], n_components=k), _records(ia, fa, bs, fp16=i == 1), 0.05, context=i == 2)
                for i, (k, bs) in enumerate([(1, 32), (5, 64), (16, 20), (9, 300), (16, 1)])]
    want = [p.buffers() for p in problems]
    for p, b in zip(problems, want):
        _single(p, b)
    got = [p.buffers() for p in problems]
    _many(problems, got)
    _assert_bitwise(problems, got, want)


def test_two_launches_give_the_same_bits():
    problems = _mixed_problems()
    first, second = [p.buffers() for p in problems], [p.buffers() for p in problems]
    _many(problems, first)
    _many(problems, second)
    _assert_bitwise(problems, second, first)


def test_together_matches_each_model_alone():
    from permutect_b200.architecture.posterior_model import learn_priors_and_spectra_together
    z, ia, fa = _golden()
    models = [_model(z, "default"), _model(z, "het_beta", 0.1, seed=7), _model(z, "no_germline"), _model(z, "default", 0.2, seed=8)]
    records = [_records(ia, fa, 16), _records(ia[:200], fa[:200], 64, fp16=True), _records(ia, fa, 7), _records(ia[10:], fa[10:], 300)]
    ratios, rates = [10.0, 5.0, 10.0, 20.0], [0.05, 0.05, 0.01, 0.05]
    alone = [copy.deepcopy(m) for m in models]
    want = [m.learn_priors_and_spectra(r, num_iterations=6, ignored_to_non_ignored_ratio=q, learning_rate=lr)
            for m, r, q, lr in zip(alone, records, ratios, rates)]
    got = learn_priors_and_spectra_together(models, records, 6, ratios, learning_rate=rates)
    assert got == want
    for i, (m, a) in enumerate(zip(models, alone)):
        assert m.priors.use_context_dependent_snv_priors and a.priors.use_context_dependent_snv_priors
        sd, sa = m.state_dict(), a.state_dict()
        assert sd.keys() == sa.keys()
        for k in sd:
            assert torch.equal(sd[k], sa[k]), f"model {i}: {k} differs"
        # the context M step ran: the SNV table is no longer one constant
        assert float(m.priors.somatic_snv_log_priors_rrra.detach()[0:4, 0:4, 0:4, 0:4].std()) > 0


def test_together_refuses_records_on_another_device():
    from permutect_b200.architecture.posterior_model import PosteriorModel, learn_priors_and_spectra_together
    z, ia, fa = _golden()
    with pytest.raises(RuntimeError, match="device"):
        learn_priors_and_spectra_together([_model(z, "default"), PosteriorModel(-3.0, -4.0, device="cpu")],
                                          [_records(ia, fa, 16), _records(ia, fa, 16)], 2, 10.0)
