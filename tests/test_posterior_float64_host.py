"""The float64 mode of the posterior oracle (oracle/posterior_model_oracle.py, ``dtype=torch.float64``), the reference
the posterior kernels are held to in test_posterior_float64_gpu.py: against scipy's binomial and beta-binomial on the
edge rows of posterior_records.edge_records, against the reference-generated golden data, and the float32 default
unchanged bit for bit.  Each check prints its worst measured error next to its tolerance."""
import os

import numpy as np
import pytest
import torch
from scipy.special import gammaln, logsumexp
from scipy.stats import betabinom, binom

from oracle import posterior_model_oracle as orc
from posterior_records import edge_records, model_state

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "posterior_model.npz")
FLOAT32_GOLDEN = os.path.join(HERE, "golden", "posterior_oracle_float32.npz")
F64 = torch.float64


def _scipy_tables(sd, ia, fa, no_germline, het_beta, context):
    """spectra_log_lks_bc, normal_log_lks_bc and log_posteriors_bc restated with scipy.stats (float64) from the
    reference's formulas (posterior_model_spectra.py, somatic_spectrum.py, artifact_spectra.py, normal_artifact_spectrum.py,
    posterior_model_priors.py)."""
    s = "spectra."
    p = {k: np.asarray(v, dtype=np.float64) for k, v in sd.items()}
    sig = lambda x: 1 / (1 + np.exp(-x))
    cf = sig(p[s + "somatic_spectrum.parametrizations.cf_k.original"])
    lw_raw = p[s + "somatic_spectrum.parametrizations.log_weights_k.original"]
    logw = lw_raw - logsumexp(lw_raw)
    art_a, art_b = (np.exp(p[s + f"artifact_spectra.parametrizations.{n}_dv.original"]) for n in ("alpha", "beta"))
    na_a, na_b = (np.exp(p[s + f"normal_artifact_spectra.normal_spectrum.parametrizations.{n}_dv.original"]) for n in ("alpha", "beta"))
    mult = sig(p[s + "normal_artifact_spectra.parametrizations.mean_multiplier_v.original"])
    conc = np.exp(p[s + "normal_artifact_spectra.parametrizations.concentration_v.original"])
    vt = ia[:, 3].astype(int)
    n, k, nn, nk = (ia[:, i].astype(np.float64) for i in (5, 6, 7, 8))
    f = fa.astype(np.float64)
    af, maf, nmaf, logit = f[:, 2], f[:, 3], f[:, 4], f[:, 5]
    t = 0.001 + 0.01 * np.arange(100)
    mc = np.minimum(maf, 0.49)[:, None, None]
    pk = (1 - mc) * cf[None, :, None] * t + mc * cf[None, :, None] * (1 - t)            # [B, K, 100]
    ub = logsumexp(binom.logpmf(k[:, None, None], n[:, None, None], pk), axis=2) - np.log(100)
    som = np.logaddexp(p[s + "somatic_spectrum.log_non_background_weight"] + logsumexp(logw + ub, axis=1),
                       p[s + "somatic_spectrum.log_background_weight"] + betabinom.logpmf(
                           k, n, p[s + "somatic_spectrum.background_alpha"], p[s + "somatic_spectrum.background_beta"]))
    db = (n >= 10).astype(int) + (n >= 20).astype(int)
    ndb = (nn >= 10).astype(int) + (nn >= 20).astype(int)
    a_b = 0.001 + nk / (nn + 0.001) * mult[vt] * conc[vt]
    b_b = np.maximum(conc[vt] - a_b, 0.001)

    def germ(ma, kk, nd):
        het, hom = 2 * af * (1 - af), af * af
        hp = het / (het + hom)
        if het_beta is None:
            minor, major = binom.logpmf(kk, nd, ma), binom.logpmf(kk, nd, 1 - ma)
        else:
            minor = major = betabinom.logpmf(kk, nd, het_beta, het_beta)
        return logsumexp(np.stack([np.log(hp / 2) + minor, np.log(hp / 2) + major,
                                   np.log(1 - hp) + betabinom.logpmf(kk, nd, 98.0, 2.0)]), axis=0)

    spec = np.stack([som, betabinom.logpmf(k, n, art_a[db, vt], art_b[db, vt]), f[:, 0], germ(maf, k, n),
                     betabinom.logpmf(k, n, a_b, b_b)], axis=1)
    norm = np.stack([f[:, 1], f[:, 1], f[:, 1], germ(nmaf, nk, nn),
                     np.where(nk < 1, -9999.0, betabinom.logpmf(nk, nn, na_a[ndb, vt], na_b[ndb, vt]))], axis=1)
    pri = p["priors.log_priors_vc"][vt].copy()
    pri[:, 2] = 0
    pri[:, 3] = -9999 if no_germline else np.log(1 - (1 - af) ** 2)
    if context:
        L = (ia.shape[1] - 16) // 2
        c = (L - 1) // 2
        h = ia[:, 16:].astype(int)
        pri[vt == 0, 0] = p["priors.somatic_snv_log_priors_rrra"][h[:, c - 1], h[:, c], h[:, c + 1], h[:, c + L]][vt == 0]
    pri = pri - logsumexp(pri, axis=1, keepdims=True)
    post = pri + spec + norm
    post[:, 1] = np.where(logit < 0, -9999.0, post[:, 1] + logit)
    post[:, 4] += logit
    return {"spectra_log_lks_bc": spec, "normal_log_lks_bc": norm, "log_posteriors_bc": post}


@pytest.mark.parametrize("K,config,kind,hap_len,fp16", [
    (1, "default", "perturbed", 21, False), (2, "no_context", "saturated", 3, True), (5, "het_beta", "perturbed", 40, True),
    (15, "het_beta_small", "saturated", 21, False), (16, "no_germline", "saturated", 3, False), (16, "default", "saturated", 21, True)])
def test_float64_oracle_matches_scipy_on_the_edge_rows(K, config, kind, hap_len, fp16):
    """~1e-12 relative, plus 16 ulp (float64) of lgamma(depth + 2) for the cancelling lgamma sums of deep rows."""
    ia, fa = edge_records(150, hap_len, fp16, seed=K)
    sd, no_germline, het_beta, context = model_state(K, config, kind, seed=K)
    got = orc.log_posterior_and_ingredients(sd, ia, fa, no_germline, het_beta, context, dtype=F64)
    want = _scipy_tables(sd, ia, fa, no_germline, het_beta, context)
    depth = np.maximum(ia[:, 5], ia[:, 7]).astype(np.float64)
    atol = (1e-12 + 16 * np.finfo(np.float64).eps * gammaln(depth + 2))[:, None]
    for name, w in want.items():
        g = got[name].numpy()
        assert g.dtype == np.float64
        excess = (np.abs(g - w) - (atol + 1e-12 * np.abs(w))) / (atol + 1e-12 * np.abs(w))
        print(f"K={K} {config} {kind} hap_len {hap_len}: {name} worst |float64 oracle - scipy| at "
              f"{float(excess.max()) + 1:.2f} of its tolerance")
        assert np.all(np.isfinite(g)) and excess.max() <= 0, (name, np.unravel_index(np.argmax(excess), excess.shape))


def _golden_case(z, tag):
    sd = {k[len(tag) + 4:]: z[k] for k in z.files if k.startswith(tag + "/sd/")}
    cfg = z[tag + "/cfg"]
    return sd, bool(cfg[0]), (None if cfg[1] < 0 else float(cfg[1])), bool(cfg[2])


@pytest.mark.parametrize("tag", ["default", "no_context", "het_beta", "no_germline"])
def test_float64_oracle_lies_within_the_row_bound_of_the_golden_data(tag):
    """The golden data (float32, from the reference) against float64: inside the row bound of test_posterior_model.py,
    2e-5 relative + 2e-4 + 8 ulp (float32) of lgamma(depth + 2).  Measured: at most 0.0242 absolute, at depth 30 000."""
    z = np.load(GOLDEN)
    sd, no_germline, het_beta, context = _golden_case(z, tag)
    got = orc.log_posterior_and_ingredients(sd, z["int_array"], z["float_array"], no_germline, het_beta, context, dtype=F64)
    depth = np.maximum(z["int_array"][:, 5], z["int_array"][:, 7]).astype(np.float64)
    atol = (2e-4 + 8 * np.finfo(np.float32).eps * gammaln(depth + 2.0))[:, None]
    for name in ("log_priors_bc", "spectra_log_lks_bc", "normal_log_lks_bc", "log_posteriors_bc"):
        want = z[f"{tag}/out/{name}"].astype(np.float64)
        tol = atol + 2e-5 * np.abs(want)
        err = np.abs(got[name].numpy() - want)
        print(f"{tag}: {name} worst |float64 - golden| {float(err.max()):.2e}, at {float((err / tol).max()):.2f} of the row bound")
        assert (err <= tol).all(), name


@pytest.mark.parametrize("tag", ["default", "no_context", "het_beta", "no_germline"])
def test_float64_loss_and_gradients_lie_within_the_float32_distance_of_the_golden_data(tag):
    """The golden loss and raw-parameter gradients (float32 autograd through the reference) against float64 autograd on
    all 300 rows, deep ones included.  Measured: loss 4.3e-6 relative, gradients 2.8e-5 of each tensor's largest entry
    at most (het_beta); held to 1e-5 and 5e-5."""
    z = np.load(GOLDEN)
    sd, no_germline, het_beta, context = _golden_case(z, tag)
    loss, _, raw = orc.negative_log_evidence_and_grads(sd, z["int_array"], z["float_array"], no_germline, het_beta, context, dtype=F64)
    assert loss.dtype == F64
    rel = abs(float(loss) - float(z[f"{tag}/loss"])) / abs(float(loss))
    worst = max(float(np.abs(g.numpy() - z[f"{tag}/grad/{n}"]).max()) / float(np.abs(g.numpy()).max()) for n, g in raw.items())
    print(f"{tag}: loss rel {rel:.2e} (tol 1e-5), gradients {worst:.2e} of each tensor's max (tol 5e-5)")
    assert rel <= 1e-5 and worst <= 5e-5


def _float32_cases():
    """The (K, config, kind, hap_len, fp16) of the stored float32 outputs."""
    return [(5, "default", "perturbed", 21, False), (16, "het_beta_small", "saturated", 3, True), (2, "no_germline", "saturated", 40, False)]


def _float32_outputs(K, config, kind, hap_len, fp16):
    ia, fa = edge_records(100, hap_len, fp16, seed=K)
    sd, no_germline, het_beta, context = model_state(K, config, kind, seed=K)
    out = {k: v.numpy() for k, v in orc.log_posterior_and_ingredients(sd, ia, fa, no_germline, het_beta, context).items()}
    loss, _, raw = orc.negative_log_evidence_and_grads(sd, ia, fa, no_germline, het_beta, context)
    out["loss"] = loss.numpy()
    out.update({"grad/" + n: g.numpy() for n, g in raw.items()})
    return out


def test_float32_default_is_unchanged():
    """The default dtype gives the bits the oracle gave before it had a dtype argument (tests/golden/posterior_oracle_float32.npz,
    written by that version).  Torch's CPU kernels may round differently on another vector ISA; there the outputs are held
    to 1e-6 relative instead."""
    z = np.load(FLOAT32_GOLDEN)
    exact = str(z["cpu_capability"]) == torch.backends.cpu.get_cpu_capability()
    for case in _float32_cases():
        tag = "_".join(str(c) for c in case)
        for name, got in _float32_outputs(*case).items():
            want = z[f"{tag}/{name}"]
            assert got.dtype == np.float32, name
            if exact:
                np.testing.assert_array_equal(got, want, err_msg=f"{tag} {name}")
            else:
                np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6, err_msg=f"{tag} {name}")
