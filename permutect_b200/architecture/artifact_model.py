"""ArtifactModel: the drop-in model surface (reference: permutect/architecture/artifact_model.py).

Same constructor, attributes, methods, state-dict keys and ``.pt`` format as the reference, so its
callers (model_training.py:151-165, filter_variants.py:292-320, prune_dataset.py) run unchanged.
``compute_batch_output`` is one call into the fused sm_100a kernels (pmt_forward); in training mode
it is recorded as a single autograd node whose backward is pmt_backward, or pmt_head_backward when no tensor upstream
of the rotation trains (calibration epochs).
"""
from typing import Optional, Tuple

import torch
from torch import Tensor, nn

from permutect_b200 import constants
from permutect_b200.architecture.layers import (MLP, Adversarial, DNASequenceConvolution, EuclideanTransformation,
                                                FeatureClustering, GatedRefAltMLP)
from permutect_b200.data.batch import Batch
from permutect_b200.data.datum import Data
from permutect_b200.engine import function as engine
from permutect_b200.engine import plan as planner
from permutect_b200.parameters import ModelParameters
from permutect_b200.sets.ragged_sets import RaggedSets
from permutect_b200.utils.enums import Epoch

MAX_OUTLIER_LOGIT = 10      # artifact_model.py:32
MAX_ALT_COUNT = 15          # count_binning.py:10


def gpu_if_available() -> torch.device:
    return torch.device("cuda" if torch.cuda.is_available() else "cpu")


class BatchOutput:
    """artifact_model.py:38-73.  All tensors come straight from the fused forward."""

    def __init__(self, features_be: Tensor, ref_features_be: Tensor, logits_b: Tensor, logits_bk: Tensor,
                 weights: Tensor, source_weights: Tensor, outlier_binary_logits: Tensor):
        self.features_be = features_be
        self.ref_features_be = ref_features_be
        self.logits_b = logits_b
        self.artifact_probs_b = torch.sigmoid(logits_b)
        self.logits_bk = logits_bk
        self.weights = weights
        self.source_weights = source_weights
        self.outlier_binary_logits = outlier_binary_logits


class BatchLosses:
    """artifact_model.py:76-90."""

    def __init__(self, supervised_losses_b, unsupervised_losses_b, alt_count_losses_b, source_prediction_losses_b,
                 total_losses_b):
        self.supervised_losses_b = supervised_losses_b
        self.unsupervised_losses_b = unsupervised_losses_b
        self.alt_count_losses_b = alt_count_losses_b
        self.source_prediction_losses_b = source_prediction_losses_b
        self.total_losses_b = total_losses_b
        self.total_loss = torch.sum(total_losses_b)


class ArtifactModel(nn.Module):
    def __init__(self, params: ModelParameters, num_read_features: int, num_info_features: int,
                 haplotypes_length: int, device=None):
        super().__init__()
        if device is None:
            device = gpu_if_available()
        self._device = torch.device(device)
        self._dtype = torch.float32
        self._haplotypes_length = haplotypes_length
        self._params = params
        if params.batch_normalize or params.dropout_p > 0:
            raise NotImplementedError("batch_normalize / dropout_p are not supported by the fused kernels")

        self.read_embedding = MLP([num_read_features] + params.read_layers)
        self.info_embedding = MLP([num_info_features] + params.info_layers)
        self.haplotypes_cnn = DNASequenceConvolution(params.ref_seq_layer_strings, haplotypes_length // 2)
        embedding_dim = (self.read_embedding.output_dimension() + self.info_embedding.output_dimension()
                         + self.haplotypes_cnn.output_dimension())
        self.ref_alt_reads_encoder = GatedRefAltMLP(d_model=embedding_dim, d_ffn=params.self_attention_hidden_dimension,
                                                    num_blocks=params.num_self_attention_layers)
        self.reducer = MLP([embedding_dim] + params.aggregation_layers)
        self.pre_clustering_transform = EuclideanTransformation(self.reducer.output_dimension())
        self.feature_clustering = FeatureClustering(feature_dimension=self.reducer.output_dimension(),
                                                    num_artifact_clusters=params.num_artifact_clusters)
        self.alt_count_predictor = Adversarial(MLP([self.reducer.output_dimension()] + [30, -1, -1, -1, 1]),
                                               adversarial_strength=0.01)
        self.alt_count_loss_func = nn.MSELoss(reduction="none")
        self.source_predictor = Adversarial(MLP([self.reducer.output_dimension()] + [1]), adversarial_strength=0.01)
        self.num_sources = 1
        self.to(device=self._device, dtype=self._dtype)
        self._desc = None
        self._loss_desc = None
        self._flat_cache = None
        self._param_list = None
        self._trunk_params = None
        self._materialization_cache = None
        self._flat_optimizer = None

    # ---- reference surface (artifact_model.py:199-230) -------------------------------------------------
    def reset_source_predictor(self, num_sources: int = 1):
        hidden = [] if num_sources == 1 else [-1, -1]
        self.source_predictor = Adversarial(MLP([self.reducer.output_dimension()] + hidden + [num_sources]),
                                            adversarial_strength=0.01).to(device=self._device, dtype=self._dtype)
        self.num_sources = num_sources
        self._desc = None
        self._loss_desc = None
        self._flat_cache = None
        self._param_list = None
        self._trunk_params = None
        self._materialization_cache = None

    def ref_alt_seq_embedding_dimension(self) -> int:
        return self.haplotypes_cnn.output_dimension()

    def haplotypes_length(self) -> int:
        return self._haplotypes_length

    def calibration_parameters(self):
        return [self.feature_clustering.parametrizations.nonartifact_stdev_e.original,
                self.feature_clustering.parametrizations.artifact_stdev_k.original]

    def set_epoch_type(self, epoch_type: Epoch):
        training = epoch_type == Epoch.TRAIN
        self.train(training)
        for p in self.parameters():
            if training:
                if p.dtype.is_floating_point:
                    p.requires_grad = True
            else:
                p.requires_grad = False

    def forward(self, batch: Batch):
        pass

    # ---- kernel plumbing -----------------------------------------------------------------------------
    def descriptor(self):
        if self._desc is None:
            self._desc = planner.build_desc(self)
        return self._desc

    def _parameter_list(self):
        """Cached list of the module's parameters (walking the module tree costs ~0.5 ms per call).  Submodules are
        only ever replaced through reset_source_predictor, which clears the cache; load_state_dict and optimisers
        update parameters in place, which the version counters below pick up."""
        if self._param_list is None:
            self._param_list = list(self.parameters())
        return self._param_list

    def _trunk_parameters(self):
        """Cached parameters of everything upstream of the rotation: read_embedding, info_embedding, haplotypes_cnn,
        ref_alt_reads_encoder and reducer (cleared with the parameter list)."""
        if self._trunk_params is None:
            self._trunk_params = [p for m in (self.read_embedding, self.info_embedding, self.haplotypes_cnn,
                                              self.ref_alt_reads_encoder, self.reducer) for p in m.parameters()]
        return self._trunk_params

    def trunk_frozen(self) -> bool:
        """True when no trunk parameter requires grad: the step trains the rotation, translation, clustering head or
        adversarial heads only (a calibration epoch), and its backward needs nothing but the forward's per-read final
        features (pmt_head_backward) instead of the whole model's backward."""
        return not any(p.requires_grad for p in self._trunk_parameters())

    def flat_weights(self) -> Tensor:
        """Materialised weights as one flat fp32 tensor.  With grad enabled this is a fresh autograd
        node (torch.cat of the constrained tensors); without grad it is cached until a parameter changes."""
        params = self._parameter_list()
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            opt = getattr(self, "_flat_optimizer", None)
            if opt is not None and opt.backs(params):
                return planner.materialize_flat(opt)          # constraint kernels on the optimiser's flat buffer
            return torch.cat([t.reshape(-1) for t in planner.materialized_tensors(self)])
        try:
            versions = tuple(p._version for p in params) + tuple(p.data_ptr() for p in params[:4])
        except RuntimeError:         # inference tensors (a model built under torch.inference_mode) track no versions
            versions = None
        if versions is None or self._flat_cache is None or self._flat_cache[0] != versions:
            with torch.no_grad():
                flat = torch.cat([t.reshape(-1) for t in planner.materialized_tensors(self)])
            if versions is None:
                self._flat_cache = None
                return flat
            self._flat_cache = (versions, flat)
        return self._flat_cache[1]

    # ---- the hot path ----------------------------------------------------------------------------------
    def calculate_features(self, batch: Batch, weight_range: float = 0) -> Tuple[RaggedSets, RaggedSets, Tensor]:
        """artifact_model.py:239-265.  ``weight_range`` is ignored, as in the reference (quirk Q3)."""
        desc = self.descriptor()
        ref_counts, alt_counts = batch.counts()
        total_ref, total_alt = int(ref_counts.sum()), int(alt_counts.sum())
        with torch.no_grad():
            out = engine.forward_call(desc, self.flat_weights(), batch, want_final=True, n_rows=total_ref + total_alt)
        final = out["final_re"]
        ref = RaggedSets(final[:total_ref], ref_counts, out["ref_means"])
        alt = RaggedSets(final[total_ref:], alt_counts, out["alt_means"])
        return ref, alt, out["info_seq"][:, desc.d_info:]

    def compute_batch_output(self, batch: Batch, balancer=None) -> BatchOutput:
        """artifact_model.py:281-297."""
        desc = self.descriptor()
        flat = self.flat_weights()
        if flat.requires_grad:
            logits_bk, alt_means, ref_means, logits_b, outlier = engine.FusedArtifactFunction.apply(flat, desc, batch,
                                                                                                    self.trunk_frozen())
        else:
            key = self._flat_cache[0] if (self._flat_cache is not None and self._flat_cache[1] is flat) else None
            out = engine.forward_call(desc, flat, batch, weights_key=key)
            logits_bk, alt_means, ref_means = out["logits_bk"], out["alt_means"], out["ref_means"]
            logits_b, outlier = out["logits_b"], out["outlier_logits"]
        if balancer is None:
            weights_b = torch.ones_like(logits_b)
            source_weights_b = torch.ones_like(logits_b)
        else:
            weights_b, source_weights_b = balancer.process_batch_and_compute_weights(
                batch, artifact_probs_b=torch.sigmoid(logits_b).detach())
        output = BatchOutput(features_be=alt_means, ref_features_be=ref_means, logits_b=logits_b, logits_bk=logits_bk,
                             weights=weights_b, source_weights=weights_b * source_weights_b,
                             outlier_binary_logits=outlier)
        output._flat = flat      # the loss head reads the same materialised weights (and shares their autograd node)
        return output

    def _loss_component(self, which: int, features_be: Tensor, batch: Batch) -> Tensor:
        """One per-variant component of the fused loss head (pmt_losses_forward; 2 = alt count, 3 = source prediction),
        differentiable w.r.t. the features and the head weights like the reference's stand-alone methods."""
        zeros = torch.zeros(batch.size(), device=self._device, dtype=self._dtype)
        return engine.FusedLossFunction.apply(self.flat_weights(), zeros, zeros, features_be, None, None,
                                              self.loss_descriptor(), batch)[which]

    def compute_source_prediction_losses(self, features_be: Tensor, batch: Batch) -> Tensor:
        """artifact_model.py:267-274."""
        return self._loss_component(3, features_be, batch)

    def compute_alt_count_losses(self, features_be: Tensor, batch: Batch) -> Tensor:
        """artifact_model.py:276-279."""
        return self._loss_component(2, features_be, batch)

    def loss_descriptor(self):
        if self._loss_desc is None or self._loss_desc[0] != (self.num_sources, float(self.alt_count_predictor.gradient_reversal.alpha),
                                                             float(self.source_predictor.gradient_reversal.alpha)):
            key = (self.num_sources, float(self.alt_count_predictor.gradient_reversal.alpha),
                   float(self.source_predictor.gradient_reversal.alpha))
            self._loss_desc = (key, planner.build_loss_desc(self, MAX_OUTLIER_LOGIT, MAX_ALT_COUNT))
        return self._loss_desc[1]

    def compute_batch_losses(self, output: BatchOutput, batch: Batch) -> BatchLosses:
        """artifact_model.py:299-325, with the adversarial heads (:267-279): one fused kernel forward, one backward."""
        flat = getattr(output, "_flat", None)
        if flat is None:
            flat = self.flat_weights()
        sup, unsup, alt_count, source, total = engine.FusedLossFunction.apply(
            flat, output.logits_b, output.outlier_binary_logits, output.features_be, output.weights, output.source_weights,
            self.loss_descriptor(), batch)
        return BatchLosses(sup, unsup, alt_count, source, total)

    # ---- persistence (artifact_model.py:327-342) -----------------------------------------------------
    def make_dict_for_saving(self, artifact_log_priors=None, artifact_spectra=None):
        return {
            constants.STATE_DICT_NAME: self.state_dict(),
            constants.HYPERPARAMS_NAME: self._params,
            constants.NUM_READ_FEATURES_NAME: self.read_embedding.input_dimension(),
            constants.NUM_INFO_FEATURES_NAME: self.info_embedding.input_dimension(),
            constants.REF_SEQUENCE_LENGTH_NAME: self.haplotypes_length(),
            constants.ARTIFACT_LOG_PRIORS_NAME: artifact_log_priors,
            constants.ARTIFACT_SPECTRA_STATE_DICT_NAME: artifact_spectra.state_dict() if artifact_spectra is not None else None,
        }

    def save_model(self, path, artifact_log_priors=None, artifact_spectra=None):
        self.reset_source_predictor()   # keeps the saved shapes stable (artifact_model.py:341)
        torch.save(self.make_dict_for_saving(artifact_log_priors, artifact_spectra), path)


def _coerce_params(hp) -> ModelParameters:
    """Accept a ModelParameters pickled by either implementation."""
    if isinstance(hp, ModelParameters):
        return hp
    return ModelParameters(read_layers=hp.read_layers, self_attention_hidden_dimension=hp.self_attention_hidden_dimension,
                           num_self_attention_layers=hp.num_self_attention_layers, info_layers=hp.info_layers,
                           aggregation_layers=hp.aggregation_layers, num_artifact_clusters=hp.num_artifact_clusters,
                           calibration_layers=hp.calibration_layers, ref_seq_layers_strings=hp.ref_seq_layer_strings,
                           dropout_p=hp.dropout_p, reweighting_range=hp.reweighting_range,
                           batch_normalize=getattr(hp, "batch_normalize", False))


def load_model(path, device: Optional[torch.device] = None):
    """artifact_model.py:345-369."""
    if device is None:
        device = gpu_if_available()
    saved = torch.load(path, map_location=device, weights_only=False)
    model = ArtifactModel(_coerce_params(saved[constants.HYPERPARAMS_NAME]),
                          num_read_features=saved[constants.NUM_READ_FEATURES_NAME],
                          num_info_features=saved[constants.NUM_INFO_FEATURES_NAME],
                          haplotypes_length=saved[constants.REF_SEQUENCE_LENGTH_NAME], device=device)
    model.load_state_dict(saved[constants.STATE_DICT_NAME])
    model.to(model._dtype)
    return model, saved[constants.ARTIFACT_LOG_PRIORS_NAME], saved[constants.ARTIFACT_SPECTRA_STATE_DICT_NAME]


class EmbeddingRecords:
    """The collector ``record_embeddings`` fills: the attributes of the reference's ``EmbeddingMetrics``
    (metrics/evaluation_metrics.py:282-289) without its TensorBoard / UMAP output, which is out of scope here.  Pass the
    reference's class instead (``metrics_factory=EmbeddingMetrics``) to get its projector output."""

    def __init__(self):
        self.label_metadata, self.correct_metadata, self.type_metadata, self.truncated_count_metadata = [], [], [], []
        self.features, self.ref_features = [], []

    def output_to_summary_writer(self, summary_writer, prefix: str = "", **kwargs):
        if summary_writer is not None and hasattr(summary_writer, "add_embedding") and self.features:
            meta = list(zip(self.label_metadata, self.correct_metadata, self.type_metadata, self.truncated_count_metadata))
            summary_writer.add_embedding(torch.vstack(self.features), metadata=meta,
                                         metadata_header=["Labels", "Correctness", "Types", "Counts"], tag=prefix + "embedding")


@torch.no_grad()
def record_embeddings(model: ArtifactModel, loader, summary_writer=None, metrics_factory=EmbeddingRecords):
    """artifact_model.py:372-408: after training, the per-variant embeddings (alt / ref set means of the final features,
    and the haplotype-CNN embedding) with their label / type / alt-count metadata.  One fused forward per batch
    (``calculate_features``); the metadata columns are read from the batch once instead of element by element.  Returns
    the two collectors (the reference returns nothing and writes them to the summary writer; both happen here)."""
    from permutect_b200.data.count_binning import alt_count_bin_index, alt_count_bin_name
    from permutect_b200.data.prefetch_generator import prefetch_generator
    from permutect_b200.utils.enums import Variation
    embedding_metrics, ref_alt_seq_metrics = metrics_factory(), metrics_factory()
    for batch in prefetch_generator(loader, model._device):
        ref_bre, alt_bre, seq_be = model.calculate_features(batch, weight_range=model._params.reweighting_range)
        alt_means_be, ref_means_be, seq_be = alt_bre.means_over_sets().cpu(), ref_bre.means_over_sets().cpu(), seq_be.cpu()
        labels_b, labeled_b = batch.get_training_labels().tolist(), batch.get_is_labeled_mask().tolist()
        labels = [("artifact" if lab > 0.5 else "non-artifact") if isl > 0.5 else "unlabeled" for lab, isl in zip(labels_b, labeled_b)]
        types = [Variation(idx).name for idx in batch.get(Data.VARIANT_TYPE).tolist()]
        counts = [alt_count_bin_name(alt_count_bin_index(ac)) for ac in batch.get(Data.ALT_COUNT).tolist()]
        for metrics, embeddings, ref_features in ((embedding_metrics, alt_means_be, ref_means_be), (ref_alt_seq_metrics, seq_be, None)):
            metrics.label_metadata.extend(labels)
            metrics.correct_metadata.extend(["unknown"] * batch.size())
            metrics.type_metadata.extend(types)
            metrics.truncated_count_metadata.extend(counts)
            metrics.features.append(embeddings)
            if ref_features is not None:
                metrics.ref_features.append(ref_features)
    embedding_metrics.output_to_summary_writer(summary_writer)
    ref_alt_seq_metrics.output_to_summary_writer(summary_writer, prefix="ref and alt allele context")
    return embedding_metrics, ref_alt_seq_metrics
