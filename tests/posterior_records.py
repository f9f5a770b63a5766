"""Posterior records and posterior models for the float64 tests of the posterior kernels
(test_posterior_float64_host.py, test_posterior_float64_gpu.py).

``edge_records`` always contains the rows where the kernels can go wrong -- depth 0, alt 0 and alt = depth, both sides of
the depth-bin edges 10 and 20, normal depth 0, depth 32 767 (the int16 limit), maf at and around the 0.49 clamp, extreme
allele frequencies, logits 0, -0 and negative, every variant type, every context code at every context position -- mixed
into random rows.  ``model_state`` gives the state dict of a posterior model with K somatic components in one of the
configurations, its raw spectra perturbed, or perturbed and pushed to saturation."""
import numpy as np
import torch

HAP_START = 16
N_FLOATS = 6
CONFIGS = {"default": (False, None, True), "no_context": (False, None, False), "het_beta": (False, 12.0, True),
           "het_beta_small": (False, 0.5, True), "no_germline": (True, None, True)}      # (no_germline, het_beta, context)


def _row(ia, i, depth, alt, ndepth, nalt, vt=None):
    ia[i, 5], ia[i, 6], ia[i, 7], ia[i, 8] = depth, alt, ndepth, nalt
    if vt is not None:
        ia[i, 3] = vt


def edge_records(n_random=400, hap_len=21, fp16=False, seed=0, max_depth=32767):
    """(int16 [B, 16 + 2 hap_len], float32 or float16 [B, 6]): the edge rows first, then n_random random rows (depths up
    to max_depth).  The float block is rounded to its type here, so the oracle and the kernel read the same values."""
    rng = np.random.default_rng(seed)
    L, c = hap_len, (hap_len - 1) // 2
    edges = []                                                    # (depth, alt, ndepth, nalt, vt or None)
    edges += [(0, 0, 0, 0, v) for v in range(5)]                  # depth 0 and normal depth 0, every type
    edges += [(50, 0, 30, 0, 0), (1, 0, 1, 0, 1), (40, 40, 25, 25, 2), (1, 1, 1, 1, 0), (2000, 2000, 300, 0, 3)]
    for d in (9, 10, 19, 20):                                     # the depth-bin edges, tumor and normal
        for v in range(5):
            edges += [(d, int(rng.integers(0, d + 1)), int(rng.integers(0, 60)), None, v)]
            nd = d
            edges += [(int(rng.integers(1, 80)), None, nd, int(rng.integers(1, nd + 1)), v)]
    edges += [(30, 5, 0, 0, 4), (30, 5, 1, 1, 0), (12, 3, 5, 1, 1), (300, 30, 0, 0, 2)]  # normal depth 0; nalt 1
    edges += [(32767, a, 32767, na, v) for a, na, v in ((0, 0, 0), (5, 1, 1), (16000, 400, 2), (32767, 32767, 3), (300, 9, 4))]
    edges += [(20000, 1, 15000, 0, 0), (32767, 1, 0, 0, 0)]
    n_edge = len(edges)
    B = n_edge + n_random
    ia = np.zeros((B, HAP_START + 2 * L), dtype=np.int16)
    fa = np.zeros((B, N_FLOATS), dtype=np.float64)
    # random rows: three quarters at depth <= 400, the rest log-uniform up to max_depth
    depth = np.where(rng.random(B) < 0.75, rng.integers(1, 401, B), np.exp(rng.uniform(np.log(400), np.log(max_depth), B)).astype(np.int64))
    depth = np.minimum(depth, max_depth)
    alt = rng.binomial(depth, rng.choice([0.002, 0.02, 0.1, 0.3, 0.5, 0.9], B))
    ndepth = np.where(rng.random(B) < 0.1, 0, rng.integers(0, 500, B))
    nalt = rng.binomial(ndepth, rng.choice([0.0, 0.01, 0.1, 0.5], B))
    ia[:, 3] = rng.integers(0, 5, B)
    ia[:, 5], ia[:, 6], ia[:, 7], ia[:, 8] = depth, alt, ndepth, nalt
    for i, (d, a, nd, na, v) in enumerate(edges):
        a = int(rng.integers(0, d + 1)) if a is None else a
        na = int(rng.integers(0, nd + 1)) if na is None else na
        _row(ia, i, d, a, nd, na, v)
    ia[:, 9] = rng.integers(0, 24, B)
    ia[:, HAP_START:] = rng.integers(0, 4, (B, 2 * L))
    # context codes: 4 at each of the four context positions of some SNVs, and every code at every position
    pos = [HAP_START + c - 1, HAP_START + c, HAP_START + c + 1, HAP_START + L + c]
    snv = np.flatnonzero(ia[:, 3] == 0)
    for j, p in enumerate(pos):
        ia[snv[j::6], p] = 4
        ia[snv[4 + j % 2::7], p] = rng.integers(0, 5, len(snv[4 + j % 2::7]))
    fa[:, 0] = -rng.uniform(0, 60, B)
    fa[:, 1] = -rng.uniform(0, 20, B)
    fa[:, 2] = 10.0 ** rng.uniform(-5, -0.005, B)
    fa[:, 3] = rng.uniform(0.0, 0.5, B)
    fa[:, 4] = rng.uniform(0.0, 0.5, B)
    fa[:, 5] = rng.normal(0, 6, B)
    ftype = np.float16 if fp16 else np.float32
    maf_edges = [0.49, float(np.nextafter(ftype(0.49), ftype(0))), 0.5]
    for i in range(n_edge):                                        # the float edges, spread over the edge rows
        fa[i, 3] = maf_edges[i % 3]
        fa[i, 4] = maf_edges[(i + 1) % 3]
        fa[i, 2] = (1e-5, 0.999, fa[i, 2])[i % 3]
        fa[i, 5] = (0.0, -0.0, -3.5, 4.0)[i % 4]
    return ia, fa.astype(ftype)


def model_state(K, config="default", kind="perturbed", seed=0):
    """(state dict of numpy float32 arrays, no_germline, het_beta, context) of a posterior model with K somatic components:
    SomaticSpectrum(K) and the default spectra with every raw tensor perturbed, log priors per type and a random SNV
    context table; kind "saturated" also sets cf_k raw +12 (and -12), a log-weight 20 above the rest and one variant
    type's concentration just above the b_b clamp."""
    from permutect_b200.architecture.posterior_model import PosteriorModel, SomaticSpectrum
    no_germline, het_beta, context = CONFIGS[config]
    model = PosteriorModel(-3.0, -4.0, no_germline_mode=no_germline, device="cpu", het_beta=het_beta)
    model.spectra.somatic_spectrum = SomaticSpectrum(K)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for t in model._raw_spectra_tensors():
            t.add_(0.3 * torch.randn(t.shape, generator=g))
        pri = model.priors.log_priors_vc
        pri[:, 0] = -3.0 + torch.rand(5, generator=g)
        pri[:, 1] = -4.0 + torch.rand(5, generator=g)
        pri[:, 4] = -5.0 + torch.rand(5, generator=g)
        model.priors.somatic_snv_log_priors_rrra.copy_(-2.0 - 10.0 * torch.rand((5, 5, 5, 5), generator=g))
        if kind == "saturated":
            s = model.spectra.somatic_spectrum.parametrizations
            s.cf_k.original[0] = 12.0
            if K > 1:
                s.cf_k.original[-1] = -12.0
                s.log_weights_k.original[K // 2] += 20.0
            na = model.spectra.normal_artifact_spectra.parametrizations
            na.concentration_v.original[2] = float(np.log(0.0025))   # b_b = max(conc - a_b, 0.001) clamps once nalt / ndepth * mult > 0.2
    sd = {k: v.detach().numpy().astype(np.float32).copy() for k, v in model.state_dict().items()}
    return sd, no_germline, het_beta, context
