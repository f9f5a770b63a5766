"""The inference half of the reference's PosteriorModel (permutect/architecture/posterior_model.py:29-99) on
libpermutect_b200: same module tree, parameter names, parametrisations and state-dict keys as the reference
(``spectra.somatic_spectrum``, ``spectra.artifact_spectra``, ``spectra.normal_artifact_spectra``, ``priors``), so a
posterior model fitted by the reference loads here and ``log_posterior_and_ingredients`` /
``posterior_probabilities_bc`` / ``error_probabilities_b`` are one kernel launch (pmt_posterior_log_posteriors).

``learn_priors_and_spectra`` (posterior_model.py:101-165) runs its E step -- negative log evidence, its gradient w.r.t.
the spectra, the posterior totals -- as pmt_posterior_fit_step and the optimiser / M step on the host; with its records
resident on the model's device (``PosteriorRecords``) every pass of the batch loop, E steps and Adam steps, is one
launch of pmt_posterior_fit_pass and only the M step stays on the host.  ``learn_priors_and_spectra_together`` fits many
samples' models side by side, a pass of all of them per launch of pmt_posterior_fit_pass_many.  Context-dependent
SNV priors are switched on for the second half of the iterations as in the reference (:125-127); its M step for them, a
PyMC ADVI fit (posterior_model_priors.py:157-203), is replaced by a deterministic fit of the same model and variational
family (architecture/snv_context_priors.py; pymc is absent from the image, so that one step has no reference golden),
on the host by default or, with ``context_fit="device"``, as one kernel launch for all models of an iteration.
``calculate_probability_thresholds`` (posterior_model.py:171-264) returns the same thresholds; its ROC plots are not
drawn.  There is no CPU path for the model itself.
"""
import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple, Union

import torch
from torch import Tensor, nn
from torch.nn import Parameter
from torch.nn.utils import parametrize

from permutect_b200.architecture.layers import BoundedNumber, LogWeights, PositiveNumber
from permutect_b200.architecture.snv_context_priors import (ContextFitPool, context_fit_inputs, fit_mutation_rates_sc,
                                                            fit_mutation_rates_sc_on_device, write_log_rates)
from permutect_b200.data.datum import HAPLOTYPES_START_IDX
from permutect_b200.engine import library as L
from permutect_b200.utils.enums import Variation

NUM_DEPTH_BINS = 3                    # spectra/artifact_spectra.py:17-18
NUM_CALLS = 5
CALL_SOMATIC, CALL_ARTIFACT, CALL_SEQ_ERROR, CALL_GERMLINE, CALL_NORMAL_ARTIFACT = range(NUM_CALLS)   # utils/enums.py Call


class SomaticSpectrum(nn.Module):
    """Parameters of spectra/somatic_spectrum.py:46-72."""

    def __init__(self, num_components: int):
        super().__init__()
        self.K = num_components
        self.cf_k = Parameter(torch.sigmoid(6 * ((torch.arange(num_components) / num_components) - 0.5)))
        parametrize.register_parametrization(self, "cf_k", BoundedNumber(0, 1))
        self.log_weights_k = Parameter(torch.log(torch.square(self.cf_k.detach())))
        parametrize.register_parametrization(self, "log_weights_k", LogWeights())
        self.log_background_weight = Parameter(torch.log(torch.tensor(0.0001)), requires_grad=False)
        self.log_non_background_weight = Parameter(torch.log(torch.tensor(1 - 0.0001)), requires_grad=False)
        self.background_alpha = Parameter(torch.tensor([1]), requires_grad=False)
        self.background_beta = Parameter(torch.tensor([1]), requires_grad=False)


class ArtifactSpectra(nn.Module):
    """Parameters of spectra/artifact_spectra.py:32-43."""

    def __init__(self):
        super().__init__()
        V = len(Variation)
        self.alpha_dv = Parameter(2 * torch.ones(NUM_DEPTH_BINS, V))
        parametrize.register_parametrization(self, "alpha_dv", PositiveNumber())
        self.beta_dv = Parameter(30 * torch.ones(NUM_DEPTH_BINS, V))
        parametrize.register_parametrization(self, "beta_dv", PositiveNumber())


class NormalArtifactSpectrum(nn.Module):
    """Parameters of spectra/normal_artifact_spectrum.py:25-36."""

    def __init__(self):
        super().__init__()
        V = len(Variation)
        self.normal_spectrum = ArtifactSpectra()
        self.mean_multiplier_v = Parameter(0.5 * torch.ones(V))
        parametrize.register_parametrization(self, "mean_multiplier_v", BoundedNumber(0, 1))
        self.concentration_v = Parameter(30 * torch.ones(V))
        parametrize.register_parametrization(self, "concentration_v", PositiveNumber())


class PosteriorModelSpectra(nn.Module):
    def __init__(self, het_beta: Optional[float] = None):
        super().__init__()
        self.het_beta = het_beta
        self.somatic_spectrum = SomaticSpectrum(num_components=5)      # spectra/posterior_model_spectra.py:74
        self.artifact_spectra = ArtifactSpectra()
        self.normal_artifact_spectra = NormalArtifactSpectrum()


class PosteriorModelPriors(nn.Module):
    """Parameters and switches of posterior_model_priors.py:68-103; the M step is PosteriorModel.update_priors_m_step."""

    def __init__(self, variant_log_prior: float, artifact_log_prior: float, no_germline_mode: bool):
        super().__init__()
        self.no_germline_mode = no_germline_mode
        self.use_context_dependent_snv_priors = True
        log_priors_vc = torch.zeros(len(Variation), NUM_CALLS)
        log_priors_vc[:, CALL_SOMATIC] = variant_log_prior
        log_priors_vc[:, CALL_ARTIFACT] = artifact_log_prior
        log_priors_vc[:, CALL_GERMLINE] = -9999 if no_germline_mode else 0
        log_priors_vc[:, CALL_NORMAL_ARTIFACT] = artifact_log_prior
        self.log_priors_vc = Parameter(log_priors_vc)
        self.somatic_snv_log_priors_rrra = Parameter(variant_log_prior * torch.ones((5, 5, 5, 5)))

    def enable_context_dependent_snv_priors(self) -> None:
        self.use_context_dependent_snv_priors = True

    def disable_context_dependent_snv_priors(self) -> None:
        self.use_context_dependent_snv_priors = False


class PosteriorModel(nn.Module):
    def __init__(self, variant_log_prior: float, artifact_log_prior: float, no_germline_mode: bool = False,
                 device=None, het_beta: Optional[float] = None):
        super().__init__()
        self._device = torch.device(device if device is not None else "cuda")
        self._dtype = torch.float32
        self.no_germline_mode = no_germline_mode
        self.het_beta = het_beta
        self.spectra = PosteriorModelSpectra(het_beta=het_beta)
        self.priors = PosteriorModelPriors(variant_log_prior, artifact_log_prior, no_germline_mode)
        self.to(device=self._device, dtype=self._dtype)

    # ---- kernel-facing view --------------------------------------------------------------------------------
    def flat_parameters(self) -> Tensor:
        """The constrained values in the order pmt_posterior_log_posteriors documents (include/permutect_b200.h)."""
        s, na = self.spectra.somatic_spectrum, self.spectra.normal_artifact_spectra
        parts = [s.cf_k, s.log_weights_k, s.log_background_weight, s.log_non_background_weight, s.background_alpha,
                 s.background_beta, self.spectra.artifact_spectra.alpha_dv, self.spectra.artifact_spectra.beta_dv,
                 na.normal_spectrum.alpha_dv, na.normal_spectrum.beta_dv, na.mean_multiplier_v, na.concentration_v,
                 self.priors.log_priors_vc, self.priors.somatic_snv_log_priors_rrra]
        with torch.no_grad():
            flat = torch.cat([p.detach().reshape(-1).to(torch.float32) for p in parts]).contiguous()
        assert flat.numel() == L.load().pmt_posterior_param_count(s.K)
        return flat

    def _inputs(self, batch):
        it, ft = batch.int_tensor, batch.float_tensor
        if it.device.type != "cuda" or ft.device != it.device:
            raise RuntimeError("PosteriorModel computes on CUDA devices only (no CPU fallback): move the batch to the GPU")
        if it.dtype != torch.int16:
            it = it.to(torch.int16)
        if ft.dtype not in (torch.float16, torch.float32):
            ft = ft.to(torch.float32)
        it, ft = it.contiguous(), ft.contiguous()
        desc = L.PmtPosteriorDesc(self.spectra.somatic_spectrum.K, HAPLOTYPES_START_IDX, (it.shape[1] - HAPLOTYPES_START_IDX) // 2,
                                  int(self.no_germline_mode), int(self.priors.use_context_dependent_snv_priors),
                                  -1.0 if self.het_beta is None else float(self.het_beta))
        return it, ft, desc, self.flat_parameters().to(it.device)

    def _run(self, batch, want: Tuple[str, ...]):
        it, ft, desc, flat = self._inputs(batch)
        B = it.shape[0]
        outs = {k: torch.empty((B, NUM_CALLS), dtype=torch.float32, device=it.device) for k in want}
        po = L.PmtPosteriorOutputs(*[outs[k].data_ptr() if k in outs else None for k in
                                     ("log_priors_bc", "spectra_log_lks_bc", "normal_log_lks_bc", "log_posteriors_bc",
                                      "posterior_probabilities_bc")])
        lib = L.load()
        L.check(lib.pmt_posterior_log_posteriors(C.byref(desc), flat.data_ptr(), it.data_ptr(), it.stride(0), ft.data_ptr(),
                                                 L.F16 if ft.dtype == torch.float16 else L.F32, ft.stride(0), B, C.byref(po),
                                                 torch.cuda.current_stream(it.device).cuda_stream))
        return outs

    # ---- reference surface (posterior_model.py:51-99) ----------------------------------------------------
    def log_posterior_and_ingredients(self, batch) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
        o = self._run(batch, ("log_priors_bc", "spectra_log_lks_bc", "normal_log_lks_bc", "log_posteriors_bc"))
        return o["log_priors_bc"], o["spectra_log_lks_bc"], o["normal_log_lks_bc"], o["log_posteriors_bc"]

    def log_relative_posteriors_bc(self, batch) -> Tensor:
        return self._run(batch, ("log_posteriors_bc",))["log_posteriors_bc"]

    def posterior_probabilities_bc(self, batch) -> Tensor:
        return self._run(batch, ("posterior_probabilities_bc",))["posterior_probabilities_bc"]

    def error_probabilities_b(self, batch, germline_mode: bool = False) -> Tensor:
        assert not (germline_mode and self.no_germline_mode), "germline mode and no-germline mode are incompatible"
        return 1 - self.posterior_probabilities_bc(batch)[:, CALL_GERMLINE if germline_mode else CALL_SOMATIC]

    @torch.no_grad()
    def calculate_probability_thresholds(self, posterior_loader, summary_writer=None, germline_mode: bool = False,
                                         recall_weight: float = 1.0):
        """posterior_model.py:171-264 without the plots: {Variation: error-probability threshold maximising F_beta}."""
        probs, types = [], []
        for batch in posterior_loader:
            probs.append(self.error_probabilities_b(batch, germline_mode))
            types.append(batch.int_tensor[:, 3].to(probs[-1].device).long())
        probs_b = torch.cat(probs) if probs else torch.zeros(0, device=self._device)
        types_b = torch.cat(types) if types else torch.zeros(0, dtype=torch.long, device=self._device)
        return {var_type: theoretical_roc_best_threshold(probs_b[types_b == int(var_type)], recall_weight)[0]
                for var_type in Variation}

    # ---- fitting (posterior_model.py:101-165) -------------------------------------------------------------
    def _spectra_tensors(self):
        s, na = self.spectra.somatic_spectrum, self.spectra.normal_artifact_spectra
        return [s.cf_k, s.log_weights_k, self.spectra.artifact_spectra.alpha_dv, self.spectra.artifact_spectra.beta_dv,
                na.normal_spectrum.alpha_dv, na.normal_spectrum.beta_dv, na.mean_multiplier_v, na.concentration_v]

    def negative_log_evidence(self, batch, posterior_totals_tc: Optional[Tensor] = None, somatic_snv_totals_rrra: Optional[Tensor] = None,
                              snv_context_totals_rrra: Optional[Tensor] = None) -> Tensor:
        """The E-step loss -mean(logsumexp(log_relative_posteriors_bc)) of :139-146 as a scalar that ``backward()`` turns
        into the same ``.grad`` of the spectra parameters as the reference's autograd; the optional buffers receive the
        E-step totals (+=) as :131-143 accumulates them."""
        it, ft, desc, flat = self._inputs(batch)
        dev = it.device
        lib = L.load()
        K = desc.n_components
        loss = torch.empty((), dtype=torch.float32, device=dev)
        grads = torch.empty(2 * K + 70, dtype=torch.float32, device=dev)
        ws = torch.empty(int(lib.pmt_posterior_fit_workspace_size(it.shape[0], K)), dtype=torch.uint8, device=dev)
        ptr = lambda t: None if t is None else t.data_ptr()
        for t in (posterior_totals_tc, somatic_snv_totals_rrra, snv_context_totals_rrra):
            assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous())
        L.check(lib.pmt_posterior_fit_step(C.byref(desc), flat.data_ptr(), it.data_ptr(), it.stride(0), ft.data_ptr(),
                                           L.F16 if ft.dtype == torch.float16 else L.F32, ft.stride(0), it.shape[0], loss.data_ptr(),
                                           grads.data_ptr(), ptr(posterior_totals_tc), ptr(somatic_snv_totals_rrra),
                                           ptr(snv_context_totals_rrra), ws.data_ptr(), ws.numel(),
                                           torch.cuda.current_stream(dev).cuda_stream))
        return _EvidenceLoss.apply(loss, grads, *self._spectra_tensors())

    def update_priors_m_step(self, posterior_totals_vc: Tensor, ignored_to_non_ignored_ratio: float,
                             somatic_snv_totals_rrra: Optional[Tensor] = None, snv_context_totals_rrra: Optional[Tensor] = None,
                             context_fit: str = "host"):
        """posterior_model_priors.py:141-224.  With context-dependent SNV priors switched on and both rrra totals given,
        ``somatic_snv_log_priors_rrra`` gets the log mutation rates of the hierarchical substitution x context model
        (snv_context_priors.context_m_step; ``context_fit="device"`` fits it on the totals' device); otherwise it is
        filled with the SNV somatic log prior (:223-225)."""
        _check_context_fit(context_fit)
        on_device = context_fit == "device"
        fit_inputs = self._m_step_before_context_fit(posterior_totals_vc, ignored_to_non_ignored_ratio, somatic_snv_totals_rrra,
                                                     snv_context_totals_rrra, on_device)
        if fit_inputs is not None:
            rates_sc = (fit_mutation_rates_sc_on_device([fit_inputs], fit_inputs[0].device)[0] if on_device
                        else fit_mutation_rates_sc(*fit_inputs))
            write_log_rates(self.priors.somatic_snv_log_priors_rrra, rates_sc)

    def _m_step_before_context_fit(self, posterior_totals_vc: Tensor, ignored_to_non_ignored_ratio: float,
                                   somatic_snv_totals_rrra: Optional[Tensor], snv_context_totals_rrra: Optional[Tensor],
                                   on_device: bool = False):
        """update_priors_m_step up to its context fit: returns that fit's inputs (snv_context_priors.context_fit_inputs, on
        the totals' device with ``on_device``) when the context-dependent SNV priors are on, else None with the M step done."""
        total_nonignored = torch.sum(posterior_totals_vc)
        overall_total = (1 + ignored_to_non_ignored_ratio) * total_nonignored
        with torch.no_grad():
            pri = self.priors
            pri.log_priors_vc.copy_(torch.log(posterior_totals_vc / (posterior_totals_vc + overall_total)))
            pri.log_priors_vc[:, CALL_SEQ_ERROR] = 0
            pri.log_priors_vc[:, CALL_GERMLINE] = -9999 if self.no_germline_mode else 0
            if pri.use_context_dependent_snv_priors:
                if somatic_snv_totals_rrra is None or snv_context_totals_rrra is None:
                    raise ValueError("context-dependent SNV priors are on: the M step needs both rrra totals")
                total_ignored_per_context = float(ignored_to_non_ignored_ratio * total_nonignored) / 64      # :150-153
                return context_fit_inputs(somatic_snv_totals_rrra, snv_context_totals_rrra, total_ignored_per_context, on_device)
            pri.somatic_snv_log_priors_rrra.fill_(pri.log_priors_vc[int(Variation.SNV), CALL_SOMATIC])
            return None

    def learn_priors_and_spectra(self, posterior_loader, num_iterations, ignored_to_non_ignored_ratio: float, summary_writer=None,
                                 learning_rate: float = 0.001, context_fit: str = "host"):
        """posterior_model.py:101-165: Adam on the spectra against the negative log evidence (E step, one kernel per
        batch), then the priors' M step; context-dependent SNV priors from the second half of the iterations on.
        ``posterior_loader`` yields batches of posterior records on the model's device; a ``PosteriorRecords`` there has
        every pass run as one kernel (``_learn_on_device``).  ``context_fit``: where the M step's context fit runs,
        "host" (float64 L-BFGS on the CPU) or "device" (pmt_snv_context_fit_many on the records' device; the same method,
        fitted rates equal to rounding).  Returns the mean loss of every iteration."""
        _check_context_fit(context_fit)
        if isinstance(posterior_loader, PosteriorRecords) and _same_device(posterior_loader.device, self._device):
            return self._learn_on_device(posterior_loader, num_iterations, ignored_to_non_ignored_ratio, summary_writer, learning_rate,
                                         context_fit)
        optimizer = torch.optim.Adam(self.spectra.parameters(), lr=learning_rate)
        self.priors.disable_context_dependent_snv_priors()
        history = []
        for epoch in range(1, num_iterations + 1):
            if epoch > (num_iterations / 2):
                self.priors.enable_context_dependent_snv_priors()
            totals_tc = torch.zeros((len(Variation), NUM_CALLS), device=self._device)
            somatic_snv_rrra = torch.zeros((5, 5, 5, 5), device=self._device)
            snv_context_rrra = torch.zeros((5, 5, 5, 5), device=self._device)
            loss_sum = torch.zeros((), device=self._device)
            count = 0
            for batch in posterior_loader:
                loss = self.negative_log_evidence(batch, totals_tc, somatic_snv_rrra, snv_context_rrra)
                optimizer.zero_grad(set_to_none=True)          # misc_utils.backpropagate (:125-129) without parameters to clip
                loss.backward()
                optimizer.step()
                loss_sum += loss.detach() * batch.size()
                count += batch.size()
            self.update_priors_m_step(totals_tc, ignored_to_non_ignored_ratio, somatic_snv_rrra, snv_context_rrra, context_fit)
            history.append(float(loss_sum) / max(count, 1))
            if summary_writer is not None:
                summary_writer.add_scalar("spectrum negative log evidence", history[-1], epoch)
        return history

    def _raw_spectra_tensors(self):
        """The raw (unconstrained) tensors behind ``_spectra_tensors``, in the same order."""
        s, na = self.spectra.somatic_spectrum, self.spectra.normal_artifact_spectra
        art, nart = self.spectra.artifact_spectra, na.normal_spectrum
        return [s.parametrizations.cf_k.original, s.parametrizations.log_weights_k.original, art.parametrizations.alpha_dv.original,
                art.parametrizations.beta_dv.original, nart.parametrizations.alpha_dv.original, nart.parametrizations.beta_dv.original,
                na.parametrizations.mean_multiplier_v.original, na.parametrizations.concentration_v.original]

    def _learn_on_device(self, records: "PosteriorRecords", num_iterations, ignored_to_non_ignored_ratio: float, summary_writer,
                         learning_rate: float, context_fit: str = "host"):
        """learn_priors_and_spectra with one pmt_posterior_fit_pass per iteration: the batches of ``records`` in order,
        each an E step and an Adam step of the raw spectra (the loop's fresh optimiser: zero moments, step 0, in flat
        device buffers for the call), then the same M step.  The raw parameters go back into the module after every pass."""
        lib = L.load()
        fit = _DeviceFit(self, records, learning_rate)
        ws = torch.empty(int(lib.pmt_posterior_fit_pass_workspace_size(self.spectra.somatic_spectrum.K)), dtype=torch.uint8,
                         device=records.device)
        stream = torch.cuda.current_stream(records.device).cuda_stream
        for epoch in range(1, num_iterations + 1):
            p = fit.begin_pass(epoch, num_iterations)
            L.check(lib.pmt_posterior_fit_pass(C.byref(p.desc), p.params, p.raw_params, p.adam_m, p.adam_v, p.adam_step, p.learning_rate,
                                               p.int_array, p.int_stride, p.float_array, p.float_kind, p.float_stride, p.n_records,
                                               p.batch_size, p.batch_losses_out, p.posterior_totals_tc, p.somatic_snv_totals_rrra,
                                               p.snv_context_totals_rrra, ws.data_ptr(), ws.numel(), stream))
            fit.end_pass()
            self.update_priors_m_step(fit.totals_tc, ignored_to_non_ignored_ratio, fit.somatic_snv_rrra, fit.snv_context_rrra,
                                      context_fit)
            fit.record(epoch, summary_writer)
        return fit.history


class _DeviceFit:
    """One model's fit on a ``PosteriorRecords`` on its device, as ``pmt_posterior_fit_pass`` and
    ``pmt_posterior_fit_pass_many`` run it: the raw spectra and the fresh optimiser's state (zero moments, step 0) in flat
    device buffers carried from pass to pass, each pass's E-step totals, and the host steps around a pass."""

    def __init__(self, model: PosteriorModel, records: "PosteriorRecords", learning_rate: float):
        dev = records.device
        self.model, self.records, self.learning_rate = model, records, float(learning_rate)
        self.raws = model._raw_spectra_tensors()
        with torch.no_grad():
            self.raw = torch.cat([t.detach().reshape(-1) for t in self.raws]).to(torch.float32).contiguous()
        self.adam_m, self.adam_v = torch.zeros_like(self.raw), torch.zeros_like(self.raw)
        self.adam_step = torch.zeros(1, dtype=torch.int64, device=dev)
        n_batches = len(records)
        self.losses = torch.empty(n_batches, dtype=torch.float32, device=dev)
        self.sizes = torch.full((n_batches,), float(records.batch_size), dtype=torch.float64, device=dev)
        self.sizes[-1] = records.size() - (n_batches - 1) * records.batch_size
        self.history = []
        model.priors.disable_context_dependent_snv_priors()

    def begin_pass(self, epoch: int, num_iterations: int) -> L.PmtPosteriorFitProblem:
        """Context-dependent SNV priors from the second half of the iterations on (:125-127), zeroed totals; returns the
        pass's arguments, valid until the next begin_pass."""
        if epoch > (num_iterations / 2):
            self.model.priors.enable_context_dependent_snv_priors()
        dev = self.records.device
        self.totals_tc = torch.zeros((len(Variation), NUM_CALLS), device=dev)
        self.somatic_snv_rrra = torch.zeros((5, 5, 5, 5), device=dev)
        self.snv_context_rrra = torch.zeros((5, 5, 5, 5), device=dev)
        it, ft, desc, self.flat = self.model._inputs(self.records)
        return L.PmtPosteriorFitProblem(desc, self.flat.data_ptr(), self.raw.data_ptr(), self.adam_m.data_ptr(), self.adam_v.data_ptr(),
                                        self.adam_step.data_ptr(), self.learning_rate, it.data_ptr(), it.stride(0), ft.data_ptr(),
                                        L.F16 if ft.dtype == torch.float16 else L.F32, ft.stride(0), self.records.size(),
                                        self.records.batch_size, self.losses.data_ptr(), self.totals_tc.data_ptr(),
                                        self.somatic_snv_rrra.data_ptr(), self.snv_context_rrra.data_ptr())

    def end_pass(self) -> None:
        """The pass's raw parameters back into the module."""
        with torch.no_grad():
            off = 0
            for t in self.raws:
                t.copy_(self.raw[off:off + t.numel()].view_as(t))
                off += t.numel()

    def record(self, epoch: int, summary_writer) -> None:
        self.history.append(float((self.losses.double() * self.sizes).sum()) / self.records.size())
        if summary_writer is not None:
            summary_writer.add_scalar("spectrum negative log evidence", self.history[-1], epoch)


def _per_model(value, n: int, what: str) -> List[float]:
    if isinstance(value, (int, float)):
        return [float(value)] * n
    values = [float(v) for v in value]
    if len(values) != n:
        raise ValueError(f"{what}: {len(values)} values for {n} models")
    return values


def _check_context_fit(context_fit) -> None:
    if context_fit not in ("host", "device"):
        raise ValueError(f'context_fit must be "host" or "device", got {context_fit!r}')


def _usable_cpus() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def learn_priors_and_spectra_together(models: Sequence[PosteriorModel], records: Sequence["PosteriorRecords"], num_iterations: int,
                                      ignored_to_non_ignored_ratio: Union[float, Sequence[float]], summary_writers=None,
                                      learning_rate: Union[float, Sequence[float]] = 0.001, context_fit: str = "host") -> List[List[float]]:
    """``models[i].learn_priors_and_spectra(records[i], ...)`` for every i, the fits side by side: a cohort's samples
    (tumour / normal pairs, the folds of an evaluation) each have their own model and records, and each fit is a chain of
    Adam steps that keeps at most 16 SMs busy, so every pass over all models is ONE pmt_posterior_fit_pass_many launch with
    a cluster of CTAs per model (one CTA each from as many models as SMs on).  Between passes each model takes the M step of ``_learn_on_device``; the float64 context fits of the
    second half run in a pool of worker processes (snv_context_priors.ContextFitPool) when there are several models, or
    with ``context_fit="device"`` as one pmt_snv_context_fit_many launch per iteration for every model that needs one.
    Every model ends with the parameters, and every history equals the history, of its own ``learn_priors_and_spectra``.

    ``records[i]`` is a ``PosteriorRecords`` (its own batch size); all models and records on one CUDA device.
    ``ignored_to_non_ignored_ratio`` and ``learning_rate``: one value for all or one per model; ``summary_writers``: None
    or one writer (or None) per model.  Returns one history per model."""
    _check_context_fit(context_fit)
    on_device = context_fit == "device"
    models, records = list(models), list(records)
    n = len(models)
    if n == 0:
        raise ValueError("learn_priors_and_spectra_together: no models")
    if len(records) != n:
        raise ValueError(f"learn_priors_and_spectra_together: {n} models but {len(records)} record sets")
    ratios = _per_model(ignored_to_non_ignored_ratio, n, "ignored_to_non_ignored_ratio")
    rates = _per_model(learning_rate, n, "learning_rate")
    writers = [None] * n if summary_writers is None else list(summary_writers)
    if len(writers) != n:
        raise ValueError(f"summary_writers: {len(writers)} writers for {n} models")
    dev = records[0].device if isinstance(records[0], PosteriorRecords) else None
    for i, (m, r) in enumerate(zip(models, records)):
        if not isinstance(r, PosteriorRecords):
            raise TypeError(f"records[{i}] is a {type(r).__name__}, not a PosteriorRecords")
        if not (_same_device(r.device, dev) and _same_device(m._device, dev)):
            raise RuntimeError(f"model {i} ({m._device}) and its records ({r.device}) must be on the device of records[0] ({dev})")
    lib = L.load()
    fits = [_DeviceFit(m, r, lr) for m, r, lr in zip(models, records, rates)]
    max_k = max(m.spectra.somatic_spectrum.K for m in models)
    ws = torch.empty(int(lib.pmt_posterior_fit_pass_many_workspace_size(n, max_k)), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    workers = 1 if on_device else min(n, _usable_cpus())
    pool = ContextFitPool(workers) if workers > 1 else None
    try:
        for epoch in range(1, num_iterations + 1):
            problems = (L.PmtPosteriorFitProblem * n)(*[f.begin_pass(epoch, num_iterations) for f in fits])
            L.check(lib.pmt_posterior_fit_pass_many(problems, n, ws.data_ptr(), ws.numel(), stream))
            fit_inputs = []
            for f, ratio in zip(fits, ratios):
                f.end_pass()
                fit_inputs.append(f.model._m_step_before_context_fit(f.totals_tc, ratio, f.somatic_snv_rrra, f.snv_context_rrra,
                                                                     on_device))
            pending = [(f, x) for f, x in zip(fits, fit_inputs) if x is not None]
            if pending:
                inputs = [x for _, x in pending]
                if on_device:
                    fitted = fit_mutation_rates_sc_on_device(inputs, dev)
                elif pool is not None and len(inputs) > 1:
                    fitted = pool.map(inputs)
                else:
                    fitted = [fit_mutation_rates_sc(*x) for x in inputs]
                for (f, _), rates_sc in zip(pending, fitted):
                    write_log_rates(f.model.priors.somatic_snv_log_priors_rrra, rates_sc)
            for f, w in zip(fits, writers):
                f.record(epoch, w)
    finally:
        if pool is not None:
            pool.close()
    return [f.history for f in fits]


def _same_device(a, b) -> bool:
    a, b = torch.device(a), torch.device(b)
    if a.type != b.type:
        return False
    if a.type != "cuda":
        return a == b
    cur = torch.cuda.current_device()
    return (cur if a.index is None else a.index) == (cur if b.index is None else b.index)


def theoretical_roc_best_threshold(error_probs_b: Tensor, recall_weight: float = 1.0) -> Tuple[float, float, float]:
    """(threshold, precision, sensitivity) maximising the F_beta score of the theoretical ROC: the second output of
    get_theoretical_roc_data (metrics/plotting.py:153-190), whose Python loop over the sorted probabilities becomes one
    sort, two prefix sums and an argmax on the tensor's device (float64, like the reference's Python floats)."""
    p = torch.sort(error_probs_b.detach().double().reshape(-1)).values
    if p.numel() == 0:
        return 0, 1, 0
    beta_sqr = recall_weight ** 2
    total_artifact = p.sum() + 0.0001
    total_non_artifact = p.numel() - total_artifact + 0.0002
    art_found = total_artifact - torch.cumsum(p, dim=0)
    tp = torch.cumsum(1 - p, dim=0)
    fp = total_artifact - art_found
    sensitivity = tp / total_non_artifact
    precision = tp / (tp + fp)
    harmonic_mean = (1 + beta_sqr) * sensitivity * precision / (sensitivity + (beta_sqr * precision) + 0.0001)
    best = harmonic_mean.max()
    if not bool(best > 0):
        return 0, 1, 0
    idx = int(torch.nonzero(harmonic_mean == best)[0])          # the loop keeps the FIRST maximum (strict >)
    return float(p[idx]), float(precision[idx]), float(sensitivity[idx])


class _EvidenceLoss(torch.autograd.Function):
    """Connects the kernel's loss and its gradient w.r.t. the constrained spectra tensors to autograd, which chains the
    parametrisations (sigmoid / exp / log_softmax) down to the raw parameters."""

    @staticmethod
    def forward(ctx, loss, grads, *tensors):
        ctx.save_for_backward(grads)
        ctx.shapes = [t.shape for t in tensors]
        return loss.clone()

    @staticmethod
    def backward(ctx, d_loss):
        (grads,) = ctx.saved_tensors
        out, off = [], 0
        for shape in ctx.shapes:
            n = int(torch.Size(shape).numel())
            out.append(d_loss * grads[off:off + n].view(shape))
            off += n
        return (None, None, *out)


class PosteriorBatch:
    """The two arrays of a batch of posterior records (generate_posterior_arrays, tools/filter_variants.py) on a device."""

    def __init__(self, int_array, float_array, device=None):
        self.int_tensor = torch.as_tensor(int_array)
        self.float_tensor = torch.as_tensor(float_array)
        if device is not None:
            self.int_tensor, self.float_tensor = self.int_tensor.to(device), self.float_tensor.to(device)

    def size(self) -> int:
        return self.int_tensor.shape[0]


class PosteriorRecords:
    """Posterior records resident on one CUDA device -- int16 [n, columns] and fp16 / fp32 [n, columns] tensors, the arrays
    of generate_posterior_arrays / posterior_arrays_on_device -- served as ``PosteriorBatch`` views of ``batch_size``
    consecutive records in order (the last batch may be shorter), so it serves wherever a loader of posterior batches does.
    ``PosteriorModel.learn_priors_and_spectra`` given one on the model's device runs each pass as one kernel."""

    def __init__(self, int_array, float_array, batch_size: int = 64, device=None):
        if int(batch_size) < 1:
            raise ValueError(f"batch_size must be >= 1, got {batch_size}")
        it, ft = torch.as_tensor(int_array), torch.as_tensor(float_array)
        dev = torch.device(device) if device is not None else (it.device if it.is_cuda else torch.device("cuda"))
        if dev.type != "cuda":
            raise RuntimeError("PosteriorRecords live on a CUDA device (no CPU fallback)")
        if it.ndim != 2 or ft.ndim != 2 or it.shape[0] != ft.shape[0] or it.shape[0] == 0:
            raise ValueError(f"need int [n, columns] and float [n, columns] arrays of the same n > 0, got {tuple(it.shape)} and {tuple(ft.shape)}")
        if ft.dtype not in (torch.float16, torch.float32):
            ft = ft.to(torch.float32)
        self.int_tensor = it.to(device=dev, dtype=torch.int16).contiguous()
        self.float_tensor = ft.to(device=dev).contiguous()
        self.batch_size = int(batch_size)
        self.device = self.int_tensor.device

    @classmethod
    def from_batches(cls, pairs, batch_size: int = 64, device=None) -> "PosteriorRecords":
        """Concatenates (int array, float array) pairs -- what generate_posterior_arrays yields, host or device."""
        ints, floats = zip(*[(torch.as_tensor(i), torch.as_tensor(f)) for i, f in pairs])
        dev = torch.device(device) if device is not None else (ints[0].device if ints[0].is_cuda else torch.device("cuda"))
        return cls(torch.cat([i.to(dev) for i in ints]), torch.cat([f.to(dev) for f in floats]), batch_size, dev)

    def size(self) -> int:
        return self.int_tensor.shape[0]

    def __len__(self) -> int:
        return (self.size() + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        for start in range(0, self.size(), self.batch_size):
            yield PosteriorBatch(self.int_tensor[start:start + self.batch_size], self.float_tensor[start:start + self.batch_size])
