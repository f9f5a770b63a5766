"""pmt_posterior_fit_pass (PosteriorModel.learn_priors_and_spectra on a PosteriorRecords): one launch per pass against the
per-batch loop (pmt_posterior_fit_step + autograd + torch.optim.Adam), against a float64 Adam loop on the oracle's
gradients, and bitwise against itself.  Each check prints its worst measured error relative to its tolerance."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import posterior_model_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "posterior_model.npz")
pytestmark = pytest.mark.gpu


def _case(z, tag):
    sd = {k[len(tag) + 4:]: z[k] for k in z.files if k.startswith(tag + "/sd/")}
    cfg = z[tag + "/cfg"]
    return sd, bool(cfg[0]), (None if cfg[1] < 0 else float(cfg[1])), bool(cfg[2])


def _shallow(z):
    keep = z["int_array"][:, 5] <= 400         # rows whose fp32 lgamma rounding stays small (test_posterior_model.py)
    return z["int_array"][keep], z["float_array"][keep]


def _model(sd, no_germline, het_beta, dev):
    from permutect_b200.architecture.posterior_model import PosteriorModel
    model = PosteriorModel(-3.0, -4.0, no_germline_mode=no_germline, device=dev, het_beta=het_beta)
    model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
    return model


def _raw(model):
    return [t.detach().cpu().numpy().copy() for t in model._raw_spectra_tensors()]


def _worst_scaled(got, want):
    """max over tensors of max|got - want| / max|want|"""
    return max(float(np.abs(g - w).max()) / max(float(np.abs(w).max()), 1e-30) for g, w in zip(got, want))


def _fused_pass(model, records, lr, raw=None, m=None, v=None, step=None, totals=True):
    """One pmt_posterior_fit_pass on the model's current parameters: (batch losses, raw, m, v, step, totals_tc, snv, ctx)."""
    from permutect_b200.engine import library as L
    lib = L.load()
    dev = records.device
    if raw is None:
        raw = torch.cat([t.detach().reshape(-1) for t in model._raw_spectra_tensors()]).float().contiguous()
        m, v, step = torch.zeros_like(raw), torch.zeros_like(raw), torch.zeros(1, dtype=torch.int64, device=dev)
    K = model.spectra.somatic_spectrum.K
    ws = torch.empty(int(lib.pmt_posterior_fit_pass_workspace_size(K)), dtype=torch.uint8, device=dev)
    losses = torch.empty(len(records), device=dev)
    tc, snv, ctx = (torch.zeros(s, device=dev) for s in ((5, 5), (5, 5, 5, 5), (5, 5, 5, 5)))
    it, ft = records.int_tensor, records.float_tensor
    _, _, desc, flat = model._inputs(records)
    L.check(lib.pmt_posterior_fit_pass(C.byref(desc), flat.data_ptr(), raw.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(),
                                       float(lr), it.data_ptr(), it.stride(0), ft.data_ptr(), L.F16 if ft.dtype == torch.float16 else L.F32,
                                       ft.stride(0), records.size(), records.batch_size, losses.data_ptr(),
                                       tc.data_ptr() if totals else None, snv.data_ptr() if totals else None,
                                       ctx.data_ptr() if totals else None, ws.data_ptr(), ws.numel(),
                                       torch.cuda.current_stream(dev).cuda_stream))
    torch.cuda.synchronize(dev)
    return losses, raw, m, v, step, tc, snv, ctx


def _split(flat, like):
    out, off = [], 0
    for t in like:
        out.append(flat[off:off + t.size].reshape(t.shape))
        off += t.size
    return out


@pytest.mark.parametrize("tag", ["default", "het_beta", "no_germline"])
def test_one_batch_one_pass_matches_one_loop_step(tag):
    from permutect_b200.architecture.posterior_model import PosteriorBatch, PosteriorRecords
    z = np.load(GOLDEN)
    sd, no_germline, het_beta, context = _case(z, tag)
    ia, fa = _shallow(z)
    dev = torch.device("cuda:0")
    fused = _model(sd, no_germline, het_beta, dev)
    records = PosteriorRecords(ia, fa, batch_size=len(ia), device=dev)
    losses, raw, _, _, step, tc, snv, ctx = _fused_pass(fused, records, 0.05)

    loop = _model(sd, no_germline, het_beta, dev)
    opt = torch.optim.Adam(loop.spectra.parameters(), lr=0.05)
    want_tc, want_snv, want_ctx = (torch.zeros(s, device=dev) for s in ((5, 5), (5, 5, 5, 5), (5, 5, 5, 5)))
    loss = loop.negative_log_evidence(PosteriorBatch(ia, fa, dev), want_tc, want_snv, want_ctx)
    loss.backward()
    opt.step()
    assert int(step) == 1
    rel = abs(float(losses[0]) - float(loss.detach())) / abs(float(loss.detach()))
    got_raw = _split(raw.cpu().numpy(), _raw(loop))
    raw_err = _worst_scaled(got_raw, _raw(loop))
    # totals: relative to each table's largest entry (sums of a few hundred posteriors; the loop adds the SNV tables with atomics)
    tot_err = max(float((a - b).abs().max() / b.abs().max()) for a, b in ((tc, want_tc), (snv, want_snv), (ctx, want_ctx)))
    print(f"{tag}: loss rel {rel:.2e} (tol 2e-6), raw {raw_err:.2e} of max (tol 1e-6), totals {tot_err:.2e} of max (tol 1e-5)")
    assert rel <= 2e-6
    assert raw_err <= 1e-6
    assert tot_err <= 1e-5


def _assert_fits_agree(fused, loop, h_fused, h_loop, what):
    hist = max(abs(a - b) / abs(b) for a, b in zip(h_fused, h_loop))
    raw = _worst_scaled(_raw(fused), _raw(loop))
    pri = float((fused.priors.log_priors_vc - loop.priors.log_priors_vc).detach().abs().max())
    rrra = float((fused.priors.somatic_snv_log_priors_rrra - loop.priors.somatic_snv_log_priors_rrra).detach().abs().max())
    print(f"{what}: history rel {hist:.2e}, raw {raw:.2e} of max, log_priors_vc {pri:.2e}, snv rrra {rrra:.2e} (tol 1e-4 each)")
    assert hist <= 1e-4 and raw <= 1e-4 and pri <= 1e-4 and rrra <= 1e-4


@pytest.mark.parametrize("tag", ["default", "het_beta", "no_germline"])
def test_fit_matches_the_per_batch_loop(tag):
    from permutect_b200.architecture.posterior_model import PosteriorRecords
    z = np.load(GOLDEN)
    sd, no_germline, het_beta, _ = _case(z, tag)
    ia, fa = _shallow(z)
    if len(ia) % 16 == 0:
        ia, fa = ia[:-1], fa[:-1]                  # a partial last batch
    dev = torch.device("cuda:0")
    records = PosteriorRecords(ia, fa, batch_size=16, device=dev)
    fused, loop = _model(sd, no_germline, het_beta, dev), _model(sd, no_germline, het_beta, dev)
    h_fused = fused.learn_priors_and_spectra(records, num_iterations=15, ignored_to_non_ignored_ratio=10.0, learning_rate=0.05)
    h_loop = loop.learn_priors_and_spectra(list(records), num_iterations=15, ignored_to_non_ignored_ratio=10.0, learning_rate=0.05)
    assert len(h_fused) == 15 and fused.priors.use_context_dependent_snv_priors
    _assert_fits_agree(fused, loop, h_fused, h_loop, tag)


def test_fit_pass_follows_a_float64_adam_loop_on_the_oracle_gradients():
    from permutect_b200.architecture.posterior_model import PosteriorRecords
    z = np.load(GOLDEN)
    sd, no_germline, het_beta, context = _case(z, "default")
    ia, fa = _shallow(z)
    bs = (len(ia) + 19) // 20
    dev = torch.device("cuda:0")
    model = _model(sd, no_germline, het_beta, dev)
    model.priors.use_context_dependent_snv_priors = context
    records = PosteriorRecords(ia, fa, batch_size=bs, device=dev)
    assert len(records) == 20
    _, raw, _, _, step, _, _, _ = _fused_pass(model, records, 0.05, totals=False)
    assert int(step) == 20

    names = list(orc.SPECTRA_RAW.values())
    p = {k: np.array(sd[k], dtype=np.float64) for k in names}
    m = {k: np.zeros_like(p[k]) for k in names}
    v = {k: np.zeros_like(p[k]) for k in names}
    for t in range(1, 21):
        cur = dict(sd)
        cur.update({k: torch.from_numpy(p[k]) for k in names})
        lo, hi = (t - 1) * bs, min(t * bs, len(ia))
        _, _, g = orc.negative_log_evidence_and_grads(cur, ia[lo:hi], fa[lo:hi], no_germline, het_beta, context)
        for k in names:
            gk = g[k].double().numpy()
            m[k] = 0.9 * m[k] + 0.1 * gk
            v[k] = 0.999 * v[k] + 0.001 * gk * gk
            p[k] = p[k] - 0.05 / (1 - 0.9 ** t) * m[k] / (np.sqrt(v[k]) / np.sqrt(1 - 0.999 ** t) + 1e-8)
    want = [p[k] for k in names]
    err = _worst_scaled(_split(raw.cpu().numpy().astype(np.float64), want), want)
    print(f"20 steps against float64 Adam on the oracle: {err:.2e} of each tensor's max (tol 2e-3)")
    assert err <= 2e-3


def test_fit_is_bitwise_reproducible():
    from permutect_b200.architecture.posterior_model import PosteriorRecords
    z = np.load(GOLDEN)
    sd, no_germline, het_beta, _ = _case(z, "default")
    ia, fa = _shallow(z)
    dev = torch.device("cuda:0")
    records = PosteriorRecords(ia, fa, batch_size=16, device=dev)
    runs = []
    for _ in range(2):
        model = _model(sd, no_germline, het_beta, dev)
        hist = model.learn_priors_and_spectra(records, num_iterations=6, ignored_to_non_ignored_ratio=10.0, learning_rate=0.05)
        one = _fused_pass(model, records, 0.05)
        runs.append((hist, [t.detach().clone() for t in model.parameters()], [t.clone() for t in one]))
    (h0, p0, o0), (h1, p1, o1) = runs
    assert h0 == h1
    assert all(torch.equal(a, b) for a, b in zip(p0, p1))
    assert all(torch.equal(a, b) for a, b in zip(o0, o1))


def test_full_size_pass_matches_the_loop_on_a_prefix():
    from permutect_b200.architecture.posterior_model import PosteriorModel, PosteriorRecords
    import importlib.util
    spec = importlib.util.spec_from_file_location("time_posterior_fit", os.path.join(
        os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "time_posterior_fit.py"))
    tpf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tpf)
    dev = torch.device("cuda:0")
    it, ft = tpf.synthetic_records(1_250_000, dev)
    records = PosteriorRecords(it, ft, batch_size=64, device=dev)
    model = PosteriorModel(-10.0, -10.0, device=dev)
    model.priors.disable_context_dependent_snv_priors()
    losses, raw, *_ = _fused_pass(model, records, 0.001)
    assert len(losses) == 19_532 and bool(torch.isfinite(losses).all())
    prefix = PosteriorRecords(it[:200 * 64], ft[:200 * 64], batch_size=64, device=dev)
    fused, loop = PosteriorModel(-10.0, -10.0, device=dev), PosteriorModel(-10.0, -10.0, device=dev)
    h_fused = fused.learn_priors_and_spectra(prefix, num_iterations=1, ignored_to_non_ignored_ratio=10.0)
    h_loop = loop.learn_priors_and_spectra(list(prefix), num_iterations=1, ignored_to_non_ignored_ratio=10.0)
    _assert_fits_agree(fused, loop, h_fused, h_loop, "first 200 batches of 1.25 M records")
