"""CPU oracle for the ArtifactModel hot path.  TEST INFRASTRUCTURE ONLY.

This is a functional restatement (plain torch-CPU tensor ops, no nn.Module, no CUDA) of the
reference algorithm, written from the reference's behaviour; every function cites the reference
file:line it follows (paths relative to /root/reference).  It exists so that tests/,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs have
a checker that travels to the GPU box (the reference itself does not).  Nothing under
``permutect_b200/`` may import it.

Parity pinning: the reference's own tests hold no golden vector for this path (SURVEY.md §8c), so
the oracle is pinned against outputs of the unmodified reference run in the build container:
``tests/golden/make_golden.py`` imports /root/reference and writes ``tests/golden/*.npz``;
``tests/test_oracle_golden.py`` checks this file against those fixtures (forward values, losses
and parameter gradients).

The oracle consumes the same *state dict* the reference produces (identical key names), a
hyper-parameter mapping, and a raw batch:

    raw = dict(reads_u8=[R,12] uint8  (or reads_f=[N,F] float),   all ref rows, then all alt rows
               read_indices=None | [N'] int64                      (DownsampledBatch gather, quirk Q1)
               ref_counts=[B] int, alt_counts=[B] int, info=[B,I] float, haplotypes=[B,2L] int,
               labels=[B] int (0 artifact, 1 variant, 2 unlabeled), sources=[B] int)
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor

PACKED_BYTES = 7          # datum.py:38  NUMBER_OF_BYTES_IN_PACKED_READ
MAX_LOGIT = 20.0          # feature_clustering.py:20
MAX_OUTLIER_LOGIT = 10.0  # artifact_model.py:32
MAX_ALT_COUNT = 15        # count_binning.py:10
MIN_BOUND, MAX_BOUND = 0.01, 100.0   # feature_clustering.py:49-51, exponentially_modified_gaussian.py:14-20
LABEL_ARTIFACT, LABEL_VARIANT, LABEL_UNLABELED = 0, 1, 2   # utils/enums.py Label


# --------------------------------------------------------------------------------------
# a1: batch decode                                                          batch.py:41-62
# --------------------------------------------------------------------------------------
def decode_reads(reads_u8: np.ndarray) -> np.ndarray:
    """batch.py:51-56 with plain_text_data.py:510-511.  Bytes 0..6 unpack MSB-first to 56 {0,1}
    columns; the remaining bytes go through ``(u8 - 128) / 32`` evaluated IN uint8, i.e. it wraps
    (quirk Q2): the effective map is ((u8 + 128) & 255) / 32.  Result is fp16-exact."""
    reads_u8 = np.ascontiguousarray(reads_u8, dtype=np.uint8)
    bits = np.unpackbits(reads_u8[:, :PACKED_BYTES], axis=1).astype(np.float32)
    wrapped = (reads_u8[:, PACKED_BYTES:].astype(np.int32) + 128) & 255
    return np.hstack((bits, wrapped.astype(np.float32) / 32.0))


def one_hot_haplotypes(haplotypes: Tensor, dtype=torch.float32) -> Tensor:
    """batch.py:115-130.  [B,2L] codes -> [B,10,L]; channel 2c is 'ref has code c', 2c+1 'alt has code c'."""
    B, two_l = haplotypes.shape
    L = two_l // 2
    out = torch.zeros(B, 10, L, dtype=dtype)
    codes = haplotypes.long()
    for half in range(2):                       # 0 = ref haplotype, 1 = alt haplotype
        h = codes[:, half * L:(half + 1) * L]   # [B,L]
        for c in range(5):
            out[:, 2 * c + half, :] = (h == c).to(dtype)
    return out


# --------------------------------------------------------------------------------------
# a4: MLP / DenseSkipBlock                                                     mlp.py:8-76
# --------------------------------------------------------------------------------------
def mlp(sd: Dict[str, Tensor], prefix: str, layer_sizes: Sequence[int], x: Tensor) -> Tensor:
    """mlp.py:25-76.  ``layer_sizes`` includes the input width.  A negative entry -d is a residual
    block x + alpha * g(x), g = d x (SELU -> Linear) (mlp.py:8-22); a positive entry is a Linear
    followed by SELU unless it is the last entry of the list (mlp.py:61-62)."""
    idx = 0
    n_entries = len(layer_sizes) - 1
    for k, width in enumerate(layer_sizes[1:]):
        if width < 0:
            inner = x
            for j in range(-width):
                w = sd[f"{prefix}._model.{idx}.mlp._model.{2 * j + 1}.weight"]
                b = sd[f"{prefix}._model.{idx}.mlp._model.{2 * j + 1}.bias"]
                inner = F.linear(F.selu(inner), w, b)
            x = x + sd[f"{prefix}._model.{idx}.alpha"] * inner
            idx += 1
            continue
        x = F.linear(x, sd[f"{prefix}._model.{idx}.weight"], sd[f"{prefix}._model.{idx}.bias"])
        idx += 1
        if k < n_entries - 1:
            x = F.selu(x)
            idx += 1
    return x


# --------------------------------------------------------------------------------------
# a3: haplotype CNN                                     dna_sequence_convolution.py:29-111
# --------------------------------------------------------------------------------------
def parse_layer_string(s: str):
    tokens = s.split("/")
    return tokens[0], {k: int(v) for k, v in (t.split("=") for t in tokens[1:])}


def haplotype_cnn(sd: Dict[str, Tensor], prefix: str, layer_strings: Sequence[str], x: Tensor) -> Tensor:
    """dna_sequence_convolution.py:57-111: one torch layer per layer string, in order."""
    for i, s in enumerate(layer_strings):
        kind, kw = parse_layer_string(s)
        if kind == "convolution":
            x = F.conv1d(x, sd[f"{prefix}._model.{i}.weight"], sd[f"{prefix}._model.{i}.bias"],
                         stride=kw.get("stride", 1), padding=kw.get("padding", 0), dilation=kw.get("dilation", 1))
        elif kind == "pool":
            ks = kw["kernel_size"]
            x = F.max_pool1d(x, ks, stride=kw.get("stride", ks))
        elif kind == "selu":
            x = F.selu(x)
        elif kind == "leaky_relu":
            x = F.leaky_relu(x)
        elif kind == "flatten":
            x = x.flatten(1)
        elif kind == "linear":
            x = F.linear(x, sd[f"{prefix}._model.{i}.weight"], sd[f"{prefix}._model.{i}.bias"])
        else:
            raise ValueError(f"oracle does not model layer type {kind!r}")
    return x


# --------------------------------------------------------------------------------------
# a7: ragged segment ops                                          ragged_sets.py:43-158
# --------------------------------------------------------------------------------------
def segment_ids(lengths: Tensor) -> Tensor:
    return torch.repeat_interleave(torch.arange(len(lengths)), lengths.long())


def segment_sums(x_nf: Tensor, lengths: Tensor) -> Tensor:
    """ragged_sets.py:157-158 (torch.segment_reduce sum; empty segment -> 0)."""
    out = torch.zeros((len(lengths),) + tuple(x_nf.shape[1:]), dtype=x_nf.dtype)
    return out.index_add(0, segment_ids(lengths), x_nf)


def segment_means(x_nf: Tensor, lengths: Tensor, regularizer: Optional[Tensor] = None, weight=1e-4) -> Tensor:
    """ragged_sets.py:144-155: (sum + w*r) / (len + w)."""
    sums = segment_sums(x_nf, lengths)
    if regularizer is not None:
        sums = sums + (weight * regularizer).view(1, -1)
    return sums / (lengths.to(x_nf.dtype) + weight).view(-1, 1)


# --------------------------------------------------------------------------------------
# a6: gated ref/alt MLP block                                        gated_mlp.py:148-276
# --------------------------------------------------------------------------------------
def gated_block(sd, p: str, ref: Tensor, alt: Tensor, ref_counts: Tensor, alt_counts: Tensor):
    """gated_mlp.py:177-200 (block) and :228-251 (spatial gating unit).  LayerNorms are shared
    between the ref and alt branches (quirk Q4); proj1/proj2 are separate."""
    d_model = ref.shape[1]
    ln = lambda t: F.layer_norm(t, (d_model,), sd[f"{p}.norm.weight"], sd[f"{p}.norm.bias"])
    z_ref = F.selu(F.linear(ln(ref), sd[f"{p}.proj1_ref.weight"], sd[f"{p}.proj1_ref.bias"]))
    z_alt = F.selu(F.linear(ln(alt), sd[f"{p}.proj1_alt.weight"], sd[f"{p}.proj1_alt.bias"]))
    half = z_ref.shape[1] // 2
    ln2 = lambda t: F.layer_norm(t, (half,), sd[f"{p}.sgu.norm.weight"], sd[f"{p}.sgu.norm.bias"])
    z1_ref, z2_ref = z_ref[:, :half], ln2(z_ref[:, half:])
    z1_alt, z2_alt = z_alt[:, :half], ln2(z_alt[:, half:])
    reg_weight = torch.exp(sd[f"{p}.sgu.parametrizations.reg_weight.original"]) + 0.25   # gated_mlp.py:225-226,237
    m_ref = segment_means(z2_ref, ref_counts, sd[f"{p}.sgu.ref_regularizer"], reg_weight)
    m_alt = segment_means(z2_alt, alt_counts)
    rid, aid = segment_ids(ref_counts), segment_ids(alt_counts)
    gate_ref = z2_ref * sd[f"{p}.sgu.alpha_ref"] + 1 + (sd[f"{p}.sgu.beta_ref"] * m_ref)[rid]
    gate_alt = (z2_alt * sd[f"{p}.sgu.alpha_alt"] + 1 + (sd[f"{p}.sgu.beta_alt"] * m_alt)[aid]
                + (sd[f"{p}.sgu.gamma"] * m_ref)[aid])
    ref = ref + F.linear(z1_ref * gate_ref, sd[f"{p}.proj2_ref.weight"], sd[f"{p}.proj2_ref.bias"])
    alt = alt + F.linear(z1_alt * gate_alt, sd[f"{p}.proj2_alt.weight"], sd[f"{p}.proj2_alt.bias"])
    return ref, alt


# --------------------------------------------------------------------------------------
# a8 + constrained parameters                euclidean_transformation.py, parameterizations.py
# --------------------------------------------------------------------------------------
def bounded(x: Tensor) -> Tensor:
    """parameterizations.py:77-78 with bounds (0.01, 100)."""
    return (MAX_BOUND - MIN_BOUND) * torch.sigmoid(x) + MIN_BOUND


def rotation_matrix(sd, p: str) -> Tensor:
    """torch.nn.utils.parametrizations.orthogonal on a square Linear weight (default map
    matrix_exp, trivialisation base buffer): Q = base @ expm(A), A = tril(X,-1) - tril(X,-1)^T."""
    x = sd[f"{p}.parametrizations.weight.original"]
    a = x.tril(-1)
    q = torch.matrix_exp(a - a.transpose(-1, -2))
    base_key = f"{p}.parametrizations.weight.0.base"
    return sd[base_key] @ q if base_key in sd else q


def euclidean_transform(sd, p: str, x: Tensor) -> Tensor:
    """euclidean_transformation.py:19-20: Linear(no bias) applied to (x + t)  ->  (x + t) Q^T."""
    return (x + sd[f"{p}.translation_e"][None, :]) @ rotation_matrix(sd, f"{p}.rotation_ee").t()


# --------------------------------------------------------------------------------------
# a9: clustering head                feature_clustering.py:23-135, exponentially_modified_gaussian.py
# --------------------------------------------------------------------------------------
def logerfc(z: Tensor) -> Tensor:
    """exponentially_modified_gaussian.py:30-55: asymptotic series when z > 5 (z clipped to >= 2
    inside the series), else log(max(erfc z, 1e-12))."""
    zc = z.clamp(min=2.0)
    z2 = zc * zc
    z4 = z2 * z2
    z6 = z2 * z4
    series = -z2 - torch.log(zc * math.sqrt(math.pi)) + torch.log1p(-1 / (2 * z2) + 3 / (4 * z4) - 15 / (8 * z6))
    direct = torch.log(torch.erfc(z).clamp(min=1.0e-12))
    return torch.where(z > 5, series, direct)


def clustering_log_likelihoods(sd, p: str, alt_re: Tensor, alt_counts: Tensor) -> Tensor:
    """feature_clustering.py:82-119.  Columns: 0 nonartifact, 1 outlier (2x stdev), 2.. artifact clusters."""
    E = alt_re.shape[1]
    log2pi = math.log(2.0 * math.pi)
    sigma = bounded(sd[f"{p}.parametrizations.nonartifact_stdev_e.original"])
    tau = bounded(sd[f"{p}.parametrizations.artifact_stdev_k.original"])
    dirs = sd[f"{p}.parametrizations.artifact_directions_ke.original"]
    dirs = dirs / torch.norm(dirs, dim=-1, keepdim=True)          # parametrisation (parameterizations.py:26-27)
    unit = dirs / torch.norm(dirs, dim=-1, keepdim=True)          # and again inside the head (feature_clustering.py:24), quirk Q5
    log_w = torch.log_softmax(sd[f"{p}.parametrizations.log_cluster_weights_k.original"], dim=-1)
    mu = sd[f"{p}.artifact_emg.mu_k"]
    sig_k = bounded(sd[f"{p}.artifact_emg.parametrizations.sigma_k.original"])
    lam = bounded(sd[f"{p}.artifact_emg.parametrizations.lambda_k.original"])

    def diag_gauss(stdev):                                        # feature_clustering.py:42-46
        return -(E / 2) * log2pi - torch.sum(torch.log(stdev)) - torch.sum(torch.square(alt_re / stdev), dim=-1) / 2

    ll_non = diag_gauss(sigma[None, :])
    ll_out = diag_gauss(2 * sigma[None, :])
    par_rk = alt_re @ unit.t()                                    # feature_clustering.py:23-30
    orth_rke = alt_re[:, None, :] - par_rk[:, :, None] * unit[None, :, :]
    orth_dist = torch.norm(orth_rke, dim=-1)
    ll_orth = (-((E - 1) / 2) * log2pi - (E - 1) * torch.log(tau)[None, :]
               - torch.square(orth_dist) / (2 * torch.square(tau[None, :])))
    var = torch.square(sig_k)                                     # exponentially_modified_gaussian.py:82-89
    ll_par = (torch.log(lam / 2) + logerfc((mu + lam * var - par_rk) / (math.sqrt(2.0) * sig_k))
              + (lam / 2) * (2 * mu + lam * var - 2 * par_rk))
    per_read = torch.cat((ll_non[:, None], ll_out[:, None], ll_orth + ll_par), dim=1)
    sums = segment_sums(per_read, alt_counts)
    sums = torch.cat((sums[:, :2], sums[:, 2:] + log_w[None, :]), dim=1)
    return sums


def logits_from_log_likelihoods(ll_bk: Tensor):
    """feature_clustering.py:121-135 and artifact_model.py:62-73."""
    raw = torch.logsumexp(ll_bk[:, 2:], dim=-1) - ll_bk[:, 0]
    logits_b = MAX_LOGIT * torch.tanh(raw / MAX_LOGIT)
    non_outlier = torch.logsumexp(torch.cat((ll_bk[:, :1], ll_bk[:, 2:]), dim=-1), dim=-1)
    outlier_binary_logits = ll_bk[:, 1] - non_outlier
    return logits_b, outlier_binary_logits


# --------------------------------------------------------------------------------------
# a5: calculate_features / compute_batch_output                   artifact_model.py:239-297
# --------------------------------------------------------------------------------------
def gather_reads(raw: dict) -> Tensor:
    if raw.get("reads_f") is not None:
        reads = torch.as_tensor(np.asarray(raw["reads_f"], dtype=np.float32))
    else:
        reads = torch.from_numpy(decode_reads(raw["reads_u8"]))
    idx = raw.get("read_indices")
    if idx is not None:                                           # batch.py:458-459 (quirk Q1: indices used verbatim)
        reads = reads[torch.as_tensor(np.asarray(idx)).long()]
    return reads


def cast_state_dict(sd: Dict[str, Tensor], dtype) -> Dict[str, Tensor]:
    """The floating-point tensors of ``sd`` in ``dtype`` (a no-op, graph included, when they already are)."""
    return {k: (v.to(dtype) if v.dtype.is_floating_point else v) for k, v in sd.items()}


def forward(sd: Dict[str, Tensor], hp: dict, raw: dict, dtype=torch.float32) -> dict:
    """artifact_model.py:239-297.  Returns every BatchOutput field plus the intermediates the
    tests compare (per-read final features, info/seq embedding).  ``dtype=torch.float64`` casts the
    state dict and every input on entry, so the whole restatement runs in double precision: the
    high-precision reference the kernels are measured against."""
    sd = cast_state_dict(sd, dtype)
    ref_counts = torch.as_tensor(np.asarray(raw["ref_counts"])).long()
    alt_counts = torch.as_tensor(np.asarray(raw["alt_counts"])).long()
    total_ref = int(ref_counts.sum())
    reads = gather_reads(raw).to(dtype)
    info = torch.as_tensor(np.asarray(raw["info"], dtype=np.float32)).to(dtype)
    haps = torch.as_tensor(np.asarray(raw["haplotypes"]))

    read_emb = mlp(sd, "read_embedding", [reads.shape[1]] + list(hp["read_layers"]), reads)
    info_emb = mlp(sd, "info_embedding", [info.shape[1]] + list(hp["info_layers"]), info)
    seq_emb = haplotype_cnn(sd, "haplotypes_cnn", hp["ref_seq_layer_strings"], one_hot_haplotypes(haps, dtype))
    info_seq = torch.hstack((info_emb, seq_emb))
    per_read = torch.vstack((info_seq[segment_ids(ref_counts)], info_seq[segment_ids(alt_counts)]))
    x = torch.hstack((read_emb, per_read))
    ref, alt = x[:total_ref], x[total_ref:]
    for blk in range(hp["num_self_attention_layers"]):
        ref, alt = gated_block(sd, f"ref_alt_reads_encoder.blocks.{blk}", ref, alt, ref_counts, alt_counts)
    red_sizes = [ref.shape[1]] + list(hp["aggregation_layers"])
    ref = euclidean_transform(sd, "pre_clustering_transform", mlp(sd, "reducer", red_sizes, ref))
    alt = euclidean_transform(sd, "pre_clustering_transform", mlp(sd, "reducer", red_sizes, alt))
    ll_bk = clustering_log_likelihoods(sd, "feature_clustering", alt, alt_counts)
    logits_b, outlier_logits = logits_from_log_likelihoods(ll_bk)
    return dict(features_be=segment_means(alt, alt_counts), ref_features_be=segment_means(ref, ref_counts),
                logits_b=logits_b, logits_bk=ll_bk, outlier_binary_logits=outlier_logits,
                artifact_probs_b=torch.sigmoid(logits_b), ref_seq_emb=seq_emb, info_seq_be=info_seq,
                final_ref_re=ref, final_alt_re=alt)


# --------------------------------------------------------------------------------------
# a10: losses                           artifact_model.py:267-325, gradient_reversal/functional.py
# --------------------------------------------------------------------------------------
def reverse_gradient(x: Tensor, alpha: float) -> Tensor:
    """gradient_reversal/functional.py:6-22: identity forward, -alpha * grad backward."""
    return x * (-alpha) + (x * (1.0 + alpha)).detach()


def source_predictor_sizes(num_sources: int, feat: int) -> List[int]:
    return [feat] + ([] if num_sources == 1 else [-1, -1]) + [num_sources]     # artifact_model.py:199-201


def losses(sd, hp: dict, raw: dict, out: dict, weights: Optional[Tensor] = None,
           source_weights: Optional[Tensor] = None, num_sources: int = 1,
           source_adversarial_strength: float = 0.01, dtype=torch.float32) -> dict:
    """artifact_model.py:299-325 with :267-279.  ``dtype``: as in ``forward`` (labels, weights and the
    loss constants are cast too)."""
    sd = cast_state_dict(sd, dtype)
    labels_int = torch.as_tensor(np.asarray(raw["labels"])).long()
    alt_counts = torch.as_tensor(np.asarray(raw["alt_counts"])).long()
    labels = (1.0 * (labels_int == LABEL_ARTIFACT) + 0.5 * (labels_int == LABEL_UNLABELED)).to(dtype)   # batch.py:100-102
    is_labeled = (labels_int != LABEL_UNLABELED).to(dtype)
    B = len(labels_int)
    weights = torch.ones(B, dtype=dtype) if weights is None else weights.to(dtype)
    source_weights = weights if source_weights is None else source_weights.to(dtype)
    bce = lambda logit, target: F.binary_cross_entropy_with_logits(logit, target, reduction="none")
    supervised = is_labeled * bce(out["logits_b"], labels)
    clipped = out["outlier_binary_logits"].clamp(max=MAX_OUTLIER_LOGIT)
    unsupervised = (1 - is_labeled) * bce(clipped, torch.zeros(B, dtype=dtype))
    feats = out["features_be"]
    E = feats.shape[1]
    pred = torch.sigmoid(mlp(sd, "alt_count_predictor.wrapped_module", [E, 30, -1, -1, -1, 1],
                             reverse_gradient(feats, 0.01)).view(-1))                   # artifact_model.py:180-182,276-279
    alt_count = torch.square(pred - alt_counts.to(dtype) / MAX_ALT_COUNT)
    if num_sources > 1:                                                                # artifact_model.py:267-274
        src_logits = mlp(sd, "source_predictor.wrapped_module", source_predictor_sizes(num_sources, E),
                         reverse_gradient(feats, source_adversarial_strength))
        onehot = F.one_hot(torch.as_tensor(np.asarray(raw["sources"])).long(), num_sources).to(dtype)
        source = torch.sum(torch.square(torch.softmax(src_logits, dim=-1) - onehot), dim=-1)
    else:
        source = torch.zeros(B, dtype=dtype)
    total_b = weights * (supervised + unsupervised + alt_count) + source_weights * source
    return dict(supervised_losses_b=supervised, unsupervised_losses_b=unsupervised, alt_count_losses_b=alt_count,
                source_prediction_losses_b=source, total_losses_b=total_b, total_loss=total_b.sum())


def loss_and_grads(sd: Dict[str, Tensor], hp: dict, raw: dict, trainable: Sequence[str], dtype=torch.float32, **loss_kw):
    """Autograd through the restatement: gradient of total_loss w.r.t. the named state-dict tensors
    (what ``loss.backward()`` leaves in ``param.grad``, misc_utils.py:125-127, before clipping).
    With ``dtype=torch.float64`` the leaves, and so autograd, are double precision throughout."""
    leaf = {k: (v.detach().to(dtype).clone().requires_grad_(k in trainable) if v.dtype.is_floating_point else v)
            for k, v in sd.items()}
    out = forward(leaf, hp, raw, dtype=dtype)
    ls = losses(leaf, hp, raw, out, dtype=dtype, **loss_kw)
    names = [k for k in trainable if leaf[k].requires_grad]
    grads = torch.autograd.grad(ls["total_loss"], [leaf[k] for k in names], allow_unused=True)
    return out, ls, {k: (g if g is not None else torch.zeros_like(leaf[k])) for k, g in zip(names, grads)}


def clip_and_adamw_step(params: Dict[str, Tensor], grads: Dict[str, Tensor], state: dict, lr: float,
                        weight_decay: float = 0.01, betas=(0.9, 0.999), eps: float = 1e-8, max_norm: float = 1.0):
    """misc_utils.py:125-129: clip_grad_norm_(max_norm=1.0) then AdamW.step (torch defaults)."""
    total = torch.sqrt(sum(torch.sum(g.double() ** 2) for g in grads.values())).float()
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    state["step"] = state.get("step", 0) + 1
    t = state["step"]
    for k, g in grads.items():
        g = g * coef
        m = state.setdefault(("m", k), torch.zeros_like(g))
        v = state.setdefault(("v", k), torch.zeros_like(g))
        params[k] = params[k] * (1 - lr * weight_decay)
        m.mul_(betas[0]).add_(g, alpha=1 - betas[0])
        v.mul_(betas[1]).addcmul_(g, g, value=1 - betas[1])
        denom = (v.sqrt() / math.sqrt(1 - betas[1] ** t)) + eps
        params[k] = params[k] - (lr / (1 - betas[0] ** t)) * m / denom
    return total
