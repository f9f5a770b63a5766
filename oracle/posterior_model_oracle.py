"""CPU restatement of PosteriorModel.log_posterior_and_ingredients (test infrastructure; SURVEY §8 f3).

Follows, in torch float32 on the CPU (or in float64 with ``dtype=torch.float64``: the parameters and the float block,
fp16 or fp32, are widened exactly and every constant and intermediate is float64):
  permutect/architecture/posterior_model.py:69-99            log posteriors = priors + spectra + normal + artifact logit
  permutect/architecture/posterior_model_priors.py:22-31,121-139   context-dependent log priors, log_softmax over calls
  permutect/architecture/spectra/posterior_model_spectra.py:18-124  germline likelihood, assembly of the [B, 5] tables
  permutect/architecture/spectra/somatic_spectrum.py:74-98    K uniform-binomial components + beta-binomial background
  permutect/architecture/spectra/artifact_spectra.py:17-55    beta-binomial per (depth bin, variant type)
  permutect/architecture/spectra/normal_artifact_spectrum.py:38-58
  permutect/utils/stats_utils.py:22-41,181-198                binomial / beta-binomial / uniform-binomial log-likelihoods
  permutect/utils/math_utils.py                               add_in_log_space
Pinned to tests/golden/posterior_model.npz (tests/golden/make_posterior_model_golden.py runs the unmodified reference).
Only tests/ may import this module; the product path is pmt_posterior_log_posteriors (libpermutect_b200).
"""
import math
from typing import Dict

import numpy as np
import torch
from torch import Tensor, lgamma

SOMATIC, ARTIFACT, SEQ_ERROR, GERMLINE, NORMAL_ARTIFACT = range(5)          # utils/enums.py Call
IDX = dict(VARIANT_TYPE=3, ORIGINAL_DEPTH=5, ORIGINAL_ALT_COUNT=6, ORIGINAL_NORMAL_DEPTH=7, ORIGINAL_NORMAL_ALT_COUNT=8)
FIDX = dict(SEQ_ERROR_LOG_LK=0, NORMAL_SEQ_ERROR_LOG_LK=1, ALLELE_FREQUENCY=2, MAF=3, NORMAL_MAF=4, CACHED_ARTIFACT_LOGIT=5)
HAP_START = 16


def binomial_log_lk(n, k, p):                                                   # stats_utils.py:22-26
    return lgamma(n + 1) - lgamma(n - k + 1) - lgamma(k + 1) + k * torch.log(p) + (n - k) * torch.log(1 - p)


def beta_binomial_log_lk(n, k, alpha, beta):                                   # stats_utils.py:29-41
    comb = lgamma(n + 1) - lgamma(n - k + 1) - lgamma(k + 1)
    return (comb + lgamma(k + alpha) + lgamma(n - k + beta) + lgamma(alpha + beta) - lgamma(n + alpha + beta)
            - lgamma(alpha) - lgamma(beta))


def uniform_binomial_log_lk(n, k, x1, x2, dtype=torch.float32):                # stats_utils.py:181-198
    interp = torch.arange(start=0.001, end=0.999, step=0.01, dtype=dtype)
    p = x2.unsqueeze(-1) * interp + x1.unsqueeze(-1) * (1 - interp)
    lk = binomial_log_lk(n.unsqueeze(-1), k.unsqueeze(-1), p)
    return torch.logsumexp(lk, dim=-1) - math.log(len(interp))


def constrained(sd: Dict[str, Tensor], dtype=torch.float32) -> Dict[str, Tensor]:
    """The tensors the reference's forward sees: parametrisations applied (parameterizations.py)."""
    g = lambda k: sd[k].to(dtype) if isinstance(sd[k], Tensor) else torch.as_tensor(np.asarray(sd[k]), dtype=dtype)
    s = "spectra."
    return dict(
        cf_k=torch.sigmoid(g(s + "somatic_spectrum.parametrizations.cf_k.original")),                  # BoundedNumber(0, 1)
        log_weights_k=torch.log_softmax(g(s + "somatic_spectrum.parametrizations.log_weights_k.original"), dim=-1),
        log_bg=g(s + "somatic_spectrum.log_background_weight"), log_non_bg=g(s + "somatic_spectrum.log_non_background_weight"),
        bg_alpha=g(s + "somatic_spectrum.background_alpha"), bg_beta=g(s + "somatic_spectrum.background_beta"),
        art_alpha_dv=torch.exp(g(s + "artifact_spectra.parametrizations.alpha_dv.original")),            # PositiveNumber
        art_beta_dv=torch.exp(g(s + "artifact_spectra.parametrizations.beta_dv.original")),
        na_alpha_dv=torch.exp(g(s + "normal_artifact_spectra.normal_spectrum.parametrizations.alpha_dv.original")),
        na_beta_dv=torch.exp(g(s + "normal_artifact_spectra.normal_spectrum.parametrizations.beta_dv.original")),
        na_mean_mult_v=torch.sigmoid(g(s + "normal_artifact_spectra.parametrizations.mean_multiplier_v.original")),
        na_conc_v=torch.exp(g(s + "normal_artifact_spectra.parametrizations.concentration_v.original")),
        log_priors_vc=g("priors.log_priors_vc"), snv_log_priors_rrra=g("priors.somatic_snv_log_priors_rrra"))


def depth_bins(depths):                                                         # artifact_spectra.py:17-24
    return (depths >= 10).long() + (depths >= 20).long()


def germline_log_likelihood(afs, mafs, alt, depths, het_beta, dtype=torch.float32):   # posterior_model_spectra.py:18-58
    het_probs = 2 * afs * (1 - afs)
    hom_probs = afs * afs
    het_prop = het_probs / (het_probs + hom_probs)
    hom_prop = 1 - het_prop
    ref = depths - alt
    comb = lgamma(depths + 1) - lgamma(alt + 1) - lgamma(ref + 1)
    if het_beta is None:
        minor = comb + alt * torch.log(mafs) + ref * torch.log(1 - mafs)
        major = comb + ref * torch.log(mafs) + alt * torch.log(1 - mafs)
    else:
        hb = torch.tensor([het_beta], dtype=dtype)
        minor = major = beta_binomial_log_lk(depths, alt, hb, hb)
    half = torch.log(het_prop / 2)
    hom = torch.log(hom_prop) + beta_binomial_log_lk(depths, alt, torch.tensor([98.0], dtype=dtype),
                                                         torch.tensor([2.0], dtype=dtype))
    return torch.logsumexp(torch.vstack((half + minor, half + major, hom)), dim=0)


def log_posterior_and_ingredients(sd, int_array: np.ndarray, float_array: np.ndarray, no_germline_mode: bool = False,
                                  het_beta=None, use_context_dependent_snv_priors: bool = True, dtype=torch.float32):
    return tables(constrained(sd, dtype), int_array, float_array, no_germline_mode, het_beta, use_context_dependent_snv_priors,
                  dtype)


SPECTRA_RAW = {"cf_k": "spectra.somatic_spectrum.parametrizations.cf_k.original",
               "log_weights_k": "spectra.somatic_spectrum.parametrizations.log_weights_k.original",
               "art_alpha_dv": "spectra.artifact_spectra.parametrizations.alpha_dv.original",
               "art_beta_dv": "spectra.artifact_spectra.parametrizations.beta_dv.original",
               "na_alpha_dv": "spectra.normal_artifact_spectra.normal_spectrum.parametrizations.alpha_dv.original",
               "na_beta_dv": "spectra.normal_artifact_spectra.normal_spectrum.parametrizations.beta_dv.original",
               "na_mean_mult_v": "spectra.normal_artifact_spectra.parametrizations.mean_multiplier_v.original",
               "na_conc_v": "spectra.normal_artifact_spectra.parametrizations.concentration_v.original"}


def negative_log_evidence_and_grads(sd, int_array, float_array, no_germline_mode=False, het_beta=None,
                                    use_context_dependent_snv_priors=True, dtype=torch.float32):
    """The loss of learn_priors_and_spectra (posterior_model.py:139-146: -mean logsumexp of the log posteriors) with its
    gradients by autograd through this restatement: (loss, d/d constrained tensor, d/d raw parameter = what
    ``loss.backward()`` leaves in ``.grad`` of the spectra parameters)."""
    leaf = {k: (torch.as_tensor(np.asarray(v), dtype=dtype).clone().requires_grad_(k in SPECTRA_RAW.values())
                if not isinstance(v, Tensor) else v.detach().to(dtype).clone().requires_grad_(k in SPECTRA_RAW.values()))
            for k, v in sd.items()}
    P = constrained(leaf, dtype)
    for k in SPECTRA_RAW:
        P[k].retain_grad()
    out = tables(P, int_array, float_array, no_germline_mode, het_beta, use_context_dependent_snv_priors, dtype)
    loss = -torch.mean(torch.logsumexp(out["log_posteriors_bc"], dim=1))
    loss.backward()
    zero = lambda t: torch.zeros_like(t)
    return (loss.detach(), {k: (P[k].grad if P[k].grad is not None else zero(P[k])) for k in SPECTRA_RAW},
            {raw: (leaf[raw].grad if leaf[raw].grad is not None else zero(leaf[raw])) for raw in SPECTRA_RAW.values()})


def tables(P, int_array: np.ndarray, float_array: np.ndarray, no_germline_mode: bool = False,
           het_beta=None, use_context_dependent_snv_priors: bool = True, dtype=torch.float32):
    it = torch.as_tensor(np.asarray(int_array)).long()
    ft = torch.as_tensor(np.asarray(float_array), dtype=torch.float32).to(dtype)   # fp16 / fp32 as the kernel reads them
    B = len(it)
    vt = it[:, IDX["VARIANT_TYPE"]]
    # the counts as `dtype` (exact: int16 values); integer tensors would put lgamma and friends in the default float32
    depth, alt = it[:, IDX["ORIGINAL_DEPTH"]].to(dtype), it[:, IDX["ORIGINAL_ALT_COUNT"]].to(dtype)
    ndepth, nalt = it[:, IDX["ORIGINAL_NORMAL_DEPTH"]].to(dtype), it[:, IDX["ORIGINAL_NORMAL_ALT_COUNT"]].to(dtype)
    af, maf, nmaf = ft[:, FIDX["ALLELE_FREQUENCY"]], ft[:, FIDX["MAF"]], ft[:, FIDX["NORMAL_MAF"]]
    logit = ft[:, FIDX["CACHED_ARTIFACT_LOGIT"]]

    # ---- priors (posterior_model_priors.py:121-139) ----
    pri = P["log_priors_vc"][vt, :].clone()
    pri[:, SEQ_ERROR] = 0
    pri[:, GERMLINE] = -9999 if no_germline_mode else torch.log(1 - torch.square(1 - af))
    if use_context_dependent_snv_priors:
        L = (it.shape[1] - HAP_START) // 2
        c = (L - 1) // 2
        hap = it[:, HAP_START:]
        ctx = P["snv_log_priors_rrra"][hap[:, c - 1], hap[:, c], hap[:, c + 1], hap[:, c + L]]
        is_snv = (vt == 0).to(dtype)
        pri[:, SOMATIC] = is_snv * ctx + (1 - is_snv) * pri[:, SOMATIC]
    pri = torch.log_softmax(pri, dim=-1)

    # ---- spectra (posterior_model_spectra.py:78-124) ----
    spec_cols = [None] * 5
    mafs_bk = torch.clamp(maf, max=0.49).view(-1, 1)
    cf = P["cf_k"].view(1, -1)
    ub = uniform_binomial_log_lk(depth.view(-1, 1).expand(-1, cf.shape[1]), alt.view(-1, 1).expand(-1, cf.shape[1]),
                                 mafs_bk * cf, (1 - mafs_bk) * cf, dtype)
    non_bg = torch.logsumexp(P["log_weights_k"].view(1, -1) + ub, dim=-1)
    bg = beta_binomial_log_lk(depth, alt, P["bg_alpha"], P["bg_beta"])
    spec_cols[SOMATIC] = torch.logaddexp(P["log_non_bg"] + non_bg, P["log_bg"] + bg)          # math_utils.add_in_log_space
    db = depth_bins(depth)
    spec_cols[ARTIFACT] = beta_binomial_log_lk(depth, alt, P["art_alpha_dv"][db, vt], P["art_beta_dv"][db, vt])
    ndb = depth_bins(ndepth)
    na_normal = beta_binomial_log_lk(ndepth, nalt, P["na_alpha_dv"][ndb, vt], P["na_beta_dv"][ndb, vt])
    conc = P["na_conc_v"][vt]
    a_b = 0.001 + (nalt / (ndepth + 0.001)) * P["na_mean_mult_v"][vt] * conc
    b_b = torch.clamp(conc - a_b, min=0.001)
    spec_cols[NORMAL_ARTIFACT] = beta_binomial_log_lk(depth, alt, a_b, b_b)
    spec_cols[SEQ_ERROR] = ft[:, FIDX["SEQ_ERROR_LOG_LK"]]
    spec_cols[GERMLINE] = germline_log_likelihood(af, maf, alt, depth, het_beta, dtype)
    spec = torch.stack(spec_cols, dim=1)          # (the reference fills a zeros tensor column by column: same values)

    nse = ft[:, FIDX["NORMAL_SEQ_ERROR_LOG_LK"]]
    norm_cols = [nse, nse, nse, germline_log_likelihood(af, nmaf, nalt, ndepth, het_beta, dtype),
                 torch.where(nalt < 1, torch.tensor(-9999.0, dtype=dtype), na_normal)]
    norm = torch.stack(norm_cols, dim=1)

    post_cols = list((pri + spec + norm).unbind(dim=1))
    post_cols[ARTIFACT] = post_cols[ARTIFACT] + logit
    post_cols[NORMAL_ARTIFACT] = post_cols[NORMAL_ARTIFACT] + logit
    post_cols[ARTIFACT] = torch.where(logit < 0, torch.tensor(-9999.0, dtype=dtype), post_cols[ARTIFACT])  # posterior_model.py:90-93
    post = torch.stack(post_cols, dim=1)
    return dict(log_priors_bc=pri, spectra_log_lks_bc=spec, normal_log_lks_bc=norm, log_posteriors_bc=post,
                posterior_probabilities_bc=torch.softmax(post, dim=1),
                error_probabilities_b=1 - torch.softmax(post, dim=1)[:, SOMATIC])
