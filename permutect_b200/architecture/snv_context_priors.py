"""The context-dependent somatic-SNV prior M step of the reference's PosteriorModelPriors
(permutect/architecture/posterior_model_priors.py:157-222) without PyMC.

The reference fits, with PyMC's mean-field ADVI, the hierarchical model

    overall_rate ~ Beta(1, 1e6)
    substitution_concentration, context_concentration ~ Gamma(4, 5)          (shape, rate)
    theta_s  ~ Dirichlet(substitution_concentration * 1_12)                    12 substitutions
    theta_sc ~ Dirichlet(context_concentration * 1_16), independently per s   16 flanking-base pairs
    rate_sc  = overall_rate * 12 theta_s * 16 theta_sc
    snv_sc   ~ Binomial(total_sc, rate_sc)

to the rounded E-step totals and writes ``log E_q[rate_sc]`` (the mean of 1000 draws from the fitted Gaussian) into
``somatic_snv_log_priors_rrra``.  ADVI is a stochastic optimiser, so the reference's own result is not reproducible run to
run; here the same variational family (a diagonal Gaussian over PyMC's unconstrained coordinates: log-odds for the Beta,
log for the Gammas, PyMC's ``SimplexTransform`` for the Dirichlets, each with its log-Jacobian) is fitted to the same
ELBO with a FIXED set of quasi-random standard-normal draws (sample-average approximation), which makes the objective
deterministic and lets L-BFGS take it to its optimum; the mean of ``rate_sc`` is then taken over a second fixed set of draws.
PARITY UNPINNED for this step: pymc is absent from the build image, so no golden from the reference's M step exists; the
tests hold it to the model's own limits (large counts: rate -> snv / total; empty cells shrink to their substitution's
mean) and to the reference's index conventions (``convert_rrra_tensor_to_sc``, :39-60; the write-back loop :210-222).

Host side (float64, 194 variational means + 194 scales), like the PyMC fit it replaces: the E step that produces the two
5x5x5x5 totals is the CUDA kernel ``pmt_posterior_fit_step``.  ``fit_mutation_rates_sc_on_device`` runs the same method
-- same start, same draws, the same L-BFGS algorithm with a hand-written gradient -- for many models in one launch of
pmt_snv_context_fit_many (csrc/pmt_context_fit.cu); its results agree with the host fit's to rounding.
"""
import math
import multiprocessing
from concurrent.futures import ProcessPoolExecutor
from typing import List, Sequence, Tuple

import torch
from torch import Tensor

NUM_SUBSTITUTIONS, NUM_CONTEXTS = 12, 16
_NONTRIVIAL_S = (1, 2, 3, 4, 6, 7, 8, 9, 11, 12, 13, 14)          # ref * 4 + alt with ref != alt (:53)
_ELBO_DRAWS, _MEAN_DRAWS = 64, 1000                                 # the reference averages 1000 draws (:203)


def convert_rrra_tensor_to_sc(input_rrra: Tensor) -> Tensor:
    """[left flank, ref, right flank, alt] (5 values each, index 4 = deletion) -> [12 substitutions, 16 flank pairs]
    (posterior_model_priors.py:39-60)."""
    t = input_rrra[0:4, 0:4, 0:4, 0:4].permute(0, 2, 1, 3)           # lf, rf, ref, alt
    t = t.reshape(NUM_CONTEXTS, 16)[:, list(_NONTRIVIAL_S)]
    return t.transpose(0, 1).contiguous()


def scatter_sc_to_rrra(values_sc: Tensor, out_rrra: Tensor) -> None:
    """The write-back loop of :210-222: out[lf, ref, rf, alt] = values[substitution, lf * 4 + rf] for ref != alt; every
    other entry of ``out_rrra`` (deletion indices, ref == alt) is left as it is."""
    v = values_sc.to(out_rrra.dtype).to(out_rrra.device)
    for s, flat in enumerate(_NONTRIVIAL_S):
        ref, alt = divmod(flat, 4)
        out_rrra[0:4, ref, 0:4, alt] = v[s].view(4, 4)


def _sobol_normal(n: int, dim: int, seed: int) -> Tensor:
    u = torch.quasirandom.SobolEngine(dim, scramble=True, seed=seed).draw(n, dtype=torch.float64)
    u = u.clamp(1e-9, 1 - 1e-9)
    return math.sqrt(2.0) * torch.erfinv(2 * u - 1)


def _simplex_backward(z: Tensor) -> Tuple[Tensor, Tensor]:
    """PyMC's SimplexTransform: x = softmax([z, -sum z]); returns (log x, log|det J|) with log|det J| = log N + sum log x."""
    y = torch.cat([z, -z.sum(-1, keepdim=True)], dim=-1)
    log_x = torch.log_softmax(y, dim=-1)
    return log_x, math.log(y.shape[-1]) + log_x.sum(-1)


def _log_joint(z: Tensor, total_sc: Tensor, snv_sc: Tensor) -> Tuple[Tensor, Tensor]:
    """log p(snv | z) + log p(T(z)) + log|det J_T(z)| for a batch of unconstrained points z [n, 194]; also rate_sc [n, 12, 16]."""
    S, Cx = NUM_SUBSTITUTIONS, NUM_CONTEXTS
    z_rate, z_sub, z_ctx = z[:, 0], z[:, 1], z[:, 2]
    z_s = z[:, 3:3 + (S - 1)]
    z_sc = z[:, 3 + (S - 1):].reshape(-1, S, Cx - 1)
    # overall_rate ~ Beta(1, 1e6) through log-odds
    log_r, log_1mr = torch.nn.functional.logsigmoid(z_rate), torch.nn.functional.logsigmoid(-z_rate)
    lp = math.log(1e6) + (1e6 - 1) * log_1mr + log_r + log_1mr
    # concentrations ~ Gamma(4, rate 5) through log
    for zc in (z_sub, z_ctx):
        lp = lp + 4 * math.log(5.0) - math.lgamma(4.0) + 3 * zc - 5 * torch.exp(zc) + zc
    a_s, a_c = torch.exp(z_sub), torch.exp(z_ctx)
    log_ts, jac_s = _simplex_backward(z_s)
    lp = lp + torch.lgamma(S * a_s) - S * torch.lgamma(a_s) + (a_s - 1) * log_ts.sum(-1) + jac_s
    log_tsc, jac_sc = _simplex_backward(z_sc)
    lp = lp + S * (torch.lgamma(Cx * a_c) - Cx * torch.lgamma(a_c)) + (a_c - 1) * log_tsc.sum((-1, -2)) + jac_sc.sum(-1)
    log_rate = log_r[:, None, None] + math.log(S * Cx) + log_ts[:, :, None] + log_tsc
    log_rate = log_rate.clamp(max=-1e-12)
    log_1m = torch.log1p(-torch.exp(log_rate))
    lp = lp + (snv_sc * log_rate + (total_sc - snv_sc) * log_1m).sum((-1, -2))      # binomial coefficient is constant
    return lp, torch.exp(log_rate)


DIM = 3 + (NUM_SUBSTITUTIONS - 1) + NUM_SUBSTITUTIONS * (NUM_CONTEXTS - 1)   # 194 unconstrained coordinates
_ELBO_SEED, _MEAN_SEED = 1234, 4321


def _clamped_inputs(total_sc: Tensor, snv_sc: Tensor) -> Tuple[Tensor, Tensor]:
    total = total_sc.detach().double().cpu().reshape(NUM_SUBSTITUTIONS, NUM_CONTEXTS)
    return total, torch.minimum(snv_sc.detach().double().cpu().reshape(NUM_SUBSTITUTIONS, NUM_CONTEXTS), total)


def fit_mutation_rates_sc(total_sc: Tensor, snv_sc: Tensor, max_iter: int = 300) -> Tensor:
    """E_q[rate_sc] [12, 16] (float64, CPU) of the mean-field fit described in the module docstring.  ``total_sc`` and
    ``snv_sc`` are the integer-rounded totals the reference hands to its Binomial (:158-159)."""
    mu, log_sigma, _, _ = fit_variational_sc(total_sc, snv_sc, max_iter)
    return mean_rates_sc(mu, log_sigma, total_sc, snv_sc)


def fit_variational_sc(total_sc: Tensor, snv_sc: Tensor, max_iter: int = 300) -> Tuple[Tensor, Tensor, int, int]:
    """The host fit's variational parameters (mu [194], log_sigma [194], float64) and its L-BFGS iteration and
    objective-evaluation counts."""
    total, snv = _clamped_inputs(total_sc, snv_sc)
    dim = DIM
    # start at the smoothed maximum-likelihood point
    overall = float((snv.sum() + 1.0) / (total.sum() + 1e6))
    ts = (snv.sum(1) + 1.0) / (snv.sum() + NUM_SUBSTITUTIONS)
    tsc = (snv + 1.0) / (snv.sum(1, keepdim=True) + NUM_CONTEXTS)
    simplex_fwd = lambda x: (torch.log(x) - torch.log(x).mean(-1, keepdim=True))[..., :-1]
    mu = torch.cat([torch.tensor([math.log(overall) - math.log1p(-overall), 0.0, 0.0], dtype=torch.float64),
                    simplex_fwd(ts), simplex_fwd(tsc).reshape(-1)]).requires_grad_(True)
    log_sigma = torch.full((dim,), -2.0, dtype=torch.float64, requires_grad=True)
    eps = _sobol_normal(_ELBO_DRAWS, dim, seed=_ELBO_SEED)
    opt = torch.optim.LBFGS([mu, log_sigma], lr=1.0, max_iter=max_iter, tolerance_grad=1e-9, tolerance_change=1e-12,
                            history_size=100, line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        z = mu + torch.exp(log_sigma) * eps
        lp, _ = _log_joint(z, total, snv)
        loss = -(lp.mean() + log_sigma.sum())                     # entropy of the diagonal Gaussian up to a constant
        loss.backward()
        return loss

    opt.step(closure)
    state = opt.state[mu]
    return mu.detach(), log_sigma.detach(), int(state["n_iter"]), int(state["func_evals"])


def mean_rates_sc(mu: Tensor, log_sigma: Tensor, total_sc: Tensor, snv_sc: Tensor) -> Tensor:
    """E_q[rate_sc] [12, 16]: the mean of rate_sc over the 1000 fixed draws from the Gaussian (mu, exp(log_sigma))."""
    total, snv = _clamped_inputs(total_sc, snv_sc)
    with torch.no_grad():
        z = mu.detach().double().cpu() + torch.exp(log_sigma.detach().double().cpu()) * _sobol_normal(_MEAN_DRAWS, DIM, seed=_MEAN_SEED)
        _, rate = _log_joint(z, total, snv)
        return rate.mean(0)


def context_fit_inputs(somatic_snv_totals_rrra: Tensor, snv_context_totals_rrra: Tensor,
                       total_ignored_per_context: float, on_device: bool = False) -> Tuple[Tensor, Tensor]:
    """(total_sc, snv_sc): the E-step totals rounded as the reference rounds them for its Binomial (:158-159).  On the
    CPU, or with ``on_device`` on the totals' device: the same float64 add and rounding, so the same bits either way."""
    where = (lambda t: t) if on_device else (lambda t: t.cpu())
    total_sc = torch.round(convert_rrra_tensor_to_sc(where(snv_context_totals_rrra.detach().double())) + total_ignored_per_context)
    snv_sc = torch.round(convert_rrra_tensor_to_sc(where(somatic_snv_totals_rrra.detach().double())))
    return total_sc, snv_sc


def write_log_rates(somatic_snv_log_priors_rrra: Tensor, rates_sc: Tensor) -> None:
    with torch.no_grad():
        scatter_sc_to_rrra(torch.log(rates_sc), somatic_snv_log_priors_rrra)


def context_m_step(somatic_snv_log_priors_rrra: Tensor, somatic_snv_totals_rrra: Tensor, snv_context_totals_rrra: Tensor,
                   total_ignored_per_context: float) -> Tensor:
    """posterior_model_priors.py:157-222: rounds the totals as the reference does, fits the rates and writes their logs
    into ``somatic_snv_log_priors_rrra`` in place.  Returns the fitted rates [12, 16]."""
    rates_sc = fit_mutation_rates_sc(*context_fit_inputs(somatic_snv_totals_rrra, snv_context_totals_rrra, total_ignored_per_context))
    write_log_rates(somatic_snv_log_priors_rrra, rates_sc)
    return rates_sc


def _init_fit_worker() -> None:
    torch.set_num_threads(1)
    fit_mutation_rates_sc(torch.ones(NUM_SUBSTITUTIONS, NUM_CONTEXTS), torch.zeros(NUM_SUBSTITUTIONS, NUM_CONTEXTS), max_iter=1)


def _started() -> None:
    pass


def _fit_arrays(total_sc, snv_sc):
    return fit_mutation_rates_sc(torch.from_numpy(total_sc), torch.from_numpy(snv_sc)).numpy()


class ContextFitPool:
    """``fit_mutation_rates_sc`` for the totals of many independent models at once, in spawned worker processes.  The fit
    is an L-BFGS loop of small float64 tensor operations whose time goes to Python, so threads would serialise on the GIL;
    each worker runs one torch thread.  Every fit is deterministic CPU work on fixed Sobol draws: each result is bit for
    bit what the in-process call gives.  The workers start, and load torch's lazily imported optimiser code, as soon as
    the pool is created; ``close()`` ends them."""

    def __init__(self, n_workers: int):
        self._pool = ProcessPoolExecutor(n_workers, mp_context=multiprocessing.get_context("spawn"), initializer=_init_fit_worker)
        for _ in range(n_workers):           # a process per task submitted while none is idle: start them all now
            self._pool.submit(_started)

    def map(self, inputs: Sequence[Tuple[Tensor, Tensor]]) -> List[Tensor]:
        """[fit_mutation_rates_sc(total_sc, snv_sc) for (total_sc, snv_sc) in inputs], the fits spread over the workers."""
        totals = [t.detach().double().cpu().numpy() for t, _ in inputs]
        snvs = [s.detach().double().cpu().numpy() for _, s in inputs]
        return [torch.from_numpy(r) for r in self._pool.map(_fit_arrays, totals, snvs)]

    def close(self) -> None:
        self._pool.shutdown()


_DRAW_TABLES = {}


def draw_tables(device) -> Tuple[Tensor, Tensor]:
    """The host fit's two standard-normal tables, [64, 194] for the ELBO and [1000, 194] for the rates' mean, as
    contiguous float64 on ``device``; computed once per device."""
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if device not in _DRAW_TABLES:
        _DRAW_TABLES[device] = (_sobol_normal(_ELBO_DRAWS, DIM, seed=_ELBO_SEED).to(device).contiguous(),
                                _sobol_normal(_MEAN_DRAWS, DIM, seed=_MEAN_SEED).to(device).contiguous())
    return _DRAW_TABLES[device]


def fit_context_models_on_device(total_sc: Tensor, snv_sc: Tensor, device=None) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """The fits of n models' totals ([n, 12, 16] each) in one launch of pmt_snv_context_fit_many on ``device`` (default:
    the totals' device).  Returns, on that device, rates [n, 12, 16] (E_q[rate_sc]), mu and log_sigma [n, 194], and the
    L-BFGS iteration and objective-evaluation counts [n] (int32)."""
    from permutect_b200.engine import library as L
    dev = torch.device(device) if device is not None else total_sc.device
    if dev.type != "cuda":
        raise RuntimeError("the device context fit runs on a CUDA device (the host fit is fit_mutation_rates_sc)")
    total = total_sc.detach().to(device=dev, dtype=torch.float64).reshape(-1, NUM_SUBSTITUTIONS, NUM_CONTEXTS).contiguous()
    snv = snv_sc.detach().to(device=dev, dtype=torch.float64).reshape(-1, NUM_SUBSTITUTIONS, NUM_CONTEXTS).contiguous()
    if total.shape != snv.shape:
        raise ValueError(f"total_sc {tuple(total.shape)} and snv_sc {tuple(snv.shape)} differ")
    n = total.shape[0]
    elbo, mean = draw_tables(dev)
    rates = torch.empty((n, NUM_SUBSTITUTIONS, NUM_CONTEXTS), dtype=torch.float64, device=dev)
    mu, log_sigma = (torch.empty((n, DIM), dtype=torch.float64, device=dev) for _ in range(2))
    n_iter, func_evals = (torch.empty(n, dtype=torch.int32, device=dev) for _ in range(2))
    lib = L.load()
    ws = torch.empty(int(lib.pmt_snv_context_fit_workspace_size(max(n, 1))), dtype=torch.uint8, device=dev)
    L.check(lib.pmt_snv_context_fit_many(n, total.data_ptr(), snv.data_ptr(), elbo.data_ptr(), mean.data_ptr(), rates.data_ptr(),
                                         mu.data_ptr(), log_sigma.data_ptr(), n_iter.data_ptr(), func_evals.data_ptr(),
                                         ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream))
    return rates, mu, log_sigma, n_iter, func_evals


def fit_mutation_rates_sc_on_device(inputs: Sequence[Tuple[Tensor, Tensor]], device) -> List[Tensor]:
    """[E_q[rate_sc] of (total_sc, snv_sc) for (total_sc, snv_sc) in inputs] -- the contract of ContextFitPool.map, float64
    [12, 16] CPU tensors -- from one launch of the device fit on ``device``."""
    if len(inputs) == 0:
        return []
    total = torch.stack([t.detach().to(device=device, dtype=torch.float64).reshape(NUM_SUBSTITUTIONS, NUM_CONTEXTS) for t, _ in inputs])
    snv = torch.stack([s.detach().to(device=device, dtype=torch.float64).reshape(NUM_SUBSTITUTIONS, NUM_CONTEXTS) for _, s in inputs])
    rates = fit_context_models_on_device(total, snv, device)[0].cpu()
    return list(rates.unbind(0))
