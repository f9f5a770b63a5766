"""Translates an ArtifactModel into the kernel-facing description: a PmtModelDesc (layer programs
and offsets into a flat weight buffer) plus the list of materialised tensors that fills that buffer.

Flat layout: one slot per entry of ``model.named_parameters()``, in that order and with that shape
(SURVEY.md Appendix B).  A slot whose parameter is the ``original`` of a torch parametrisation holds
the CONSTRAINED value the reference's forward would see (bounded stdev, unit directions, log-softmax
weights, exp(reg_weight), the orthogonal rotation matrix), so autograd chains the constraint
Jacobians when the flat buffer is assembled with ``torch.cat``.
"""
from typing import Dict, List, Tuple

import torch

from permutect_b200.engine import library as L

_PARAM_TAG = ".parametrizations."


def flat_layout(model) -> Tuple[Dict[str, int], int]:
    offsets, off = {}, 0
    for name, p in model.named_parameters():
        offsets[name] = off
        off += p.numel()
    return offsets, off


def _owner_and_attr(model, name: str):
    """'a.b.parametrizations.x.original' -> (module a.b, 'x')."""
    head, tail = name.split(_PARAM_TAG)
    attr = tail.split(".")[0]
    module = model.get_submodule(head) if head else model
    return module, attr


_ROTATION_KERNEL_MAX_N = 16


class _RotationFunction(torch.autograd.Function):
    """Q = base @ exp(tril(X) - tril(X)^T) and its vector-Jacobian product as single-CTA kernels (csrc/pmt_optim.cu),
    same scaling-and-squaring recipe as the torch formulation below."""

    @staticmethod
    def forward(ctx, X, base):
        lib = L.load()
        Xc = X.detach().contiguous()
        bc = None if base is None else base.detach().contiguous()
        Q = torch.empty_like(Xc)
        L.check(lib.pmt_orthogonal_forward(Xc.data_ptr(), None if bc is None else bc.data_ptr(), Xc.shape[0], Q.data_ptr(),
                                           torch.cuda.current_stream(Xc.device).cuda_stream))
        ctx.save_for_backward(Xc, bc if bc is not None else Xc.new_empty(0))
        ctx.has_base = bc is not None
        return Q

    @staticmethod
    def backward(ctx, dQ):
        Xc, bc = ctx.saved_tensors
        lib = L.load()
        dQ = dQ.contiguous().float()
        dX = torch.empty_like(Xc)
        L.check(lib.pmt_orthogonal_backward(Xc.data_ptr(), bc.data_ptr() if ctx.has_base else None, dQ.data_ptr(), Xc.shape[0],
                                            dX.data_ptr(), torch.cuda.current_stream(Xc.device).cuda_stream))
        return dX, None


def _orthogonal_without_sync(module, attr):
    """The rotation matrix of torch's ``orthogonal`` parametrisation (matrix-exponential map, square weight) evaluated
    without ``torch.matrix_exp``: that routine picks its Pade degree from a norm it reads back on the host, i.e. it
    synchronises the device twice per training step (forward and backward).  Here: scaling and squaring with FIXED
    parameters in float64 (Taylor degree 14 of A / 2^6, six squarings), exact to fp32 rounding for ||A|| up to ~64 and
    differentiable by autograd.  Mirrors torch/nn/utils/parametrizations.py:_Orthogonal.forward.
    Returns None when the parametrisation is something else."""
    plist = getattr(getattr(module, "parametrizations", None), attr, None) if hasattr(module, "parametrizations") else None
    if plist is None or len(plist) != 1:
        return None
    orth = plist[0]
    if type(orth).__name__ != "_Orthogonal" or getattr(getattr(orth, "orthogonal_map", None), "name", "") != "matrix_exp":
        return None
    X = plist.original
    if X.dim() != 2 or X.shape[0] != X.shape[1]:
        return None
    base = getattr(orth, "base", None)
    if X.is_cuda and X.dtype == torch.float32 and X.shape[0] <= _ROTATION_KERNEL_MAX_N and (base is None or base.dtype == torch.float32):
        return _RotationFunction.apply(X, base)          # pmt_orthogonal_forward / _backward: two launches instead of ~135 ops
    Xl = X.double().tril()
    A = Xl - Xl.mT
    n = A.shape[0]
    eye = torch.eye(n, dtype=A.dtype, device=A.device)
    B = A * (2.0 ** -6)
    T = eye + B / 14.0
    for k in range(13, 0, -1):
        T = eye + (B @ T) / float(k)
    for _ in range(6):
        T = T @ T
    Q = T.to(X.dtype)
    if hasattr(orth, "base"):
        Q = orth.base @ Q
    return Q


def _materialization_recipe(model):
    """[(parameter, owner module or None, attribute)] in named_parameters() order, cached on the model (walking the
    module tree and splitting names costs ~1 ms per call).  Invalidated together with the descriptor."""
    recipe = getattr(model, "_materialization_cache", None)
    if recipe is None:
        recipe = []
        for name, p in model.named_parameters():
            if _PARAM_TAG in name:
                module, attr = _owner_and_attr(model, name)
                recipe.append((p, module, attr))
            else:
                recipe.append((p, None, None))
        model._materialization_cache = recipe
    return recipe


def materialized_tensors(model) -> List[torch.Tensor]:
    """Tensors to concatenate into the flat weight buffer (autograd-connected to the raw parameters)."""
    out = []
    for p, module, attr in _materialization_recipe(model):
        if module is None:
            out.append(p)
            continue
        out.append(_constrained_value(module, attr))
    return out


def _constrained_value(module, attr):
    t = _orthogonal_without_sync(module, attr)
    if t is None:
        t = getattr(module, attr)                   # evaluates the parametrisation
    if attr == "artifact_directions_ke":
        # the head normalises the (already unit) directions once more (feature_clustering.py:24, quirk Q5)
        t = t / torch.norm(t, dim=-1, keepdim=True)
    return t


class _ConstraintPack:
    """The parametrised tensors of a model as positions in the flat buffer, built once when a FlatAdamW attaches: the
    byte mask of the entries that belong to a constraint group and the group table of pmt_constraints_forward /
    _backward, both resident on the device, and ``rotation`` = (raw parameter, owner module, attribute, offset, size) of
    the orthogonal matrix, or None.  A parametrisation other than the reference's five is refused here."""

    def __init__(self, model, device):
        import numpy as np
        offsets, n_flat = flat_layout(model)
        groups, self.rotation = [], None
        for name, p in model.named_parameters():
            if _PARAM_TAG not in name:
                continue
            module, attr = _owner_and_attr(model, name)
            off, n = offsets[name], p.numel()
            plist = getattr(module.parametrizations, attr)
            kind = type(plist[0]).__name__ if len(plist) == 1 else "?"
            if kind == "PositiveNumber":
                groups.append((L.CONSTRAINT_EXP, off, 1, n, 0.0, 0.0))
            elif kind == "BoundedNumber":
                groups.append((L.CONSTRAINT_BOUNDED, off, 1, n, float(plist[0].size), float(plist[0].min_val)))
            elif kind == "UnitVector" and p.dim() == 2:
                twice = attr == "artifact_directions_ke"
                groups.append((L.CONSTRAINT_UNIT_TWICE if twice else L.CONSTRAINT_UNIT, off, p.shape[0], p.shape[1], 0.0, 0.0))
            elif kind == "LogWeights" and p.dim() == 1:
                groups.append((L.CONSTRAINT_LOGSOFTMAX, off, 1, n, 0.0, 0.0))
            elif (kind == "_Orthogonal" and self.rotation is None and plist[0].orthogonal_map.name == "matrix_exp"
                  and p.dim() == 2 and p.shape[0] == p.shape[1]):        # what _orthogonal_without_sync evaluates
                self.rotation = (p, module, attr, off, n)
            else:
                raise NotImplementedError(f"{name}: no constraint kernel for this parametrisation")
        mask = np.zeros(n_flat, np.uint8)
        table = np.zeros(max(len(groups), 1), dtype=[("type", "<i4"), ("off", "<i4"), ("rows", "<i4"), ("cols", "<i4"),
                                                     ("a", "<f4"), ("b", "<f4")])
        for j, (t, off, rows, cols, a, b) in enumerate(groups):
            table[j] = (t, off, rows, cols, a, b)
            mask[off:off + rows * cols] = 1
        self.mask = torch.from_numpy(mask).to(device)
        self.table, self.n_groups = torch.from_numpy(table.view(np.uint8).copy()).to(device), len(groups)
        self.anchor = torch.zeros((), device=device, requires_grad=True)      # keeps the node in the graph


class _FastMaterialize(torch.autograd.Function):
    """flat materialised weights = the optimiser's flat raw-parameter buffer with the slots of the parametrised tensors
    replaced by their constrained values: parameterizations.py's maps in one kernel (PositiveNumber: exp; BoundedNumber:
    size * sigmoid + min; UnitVector: x / |x|, applied twice for the cluster directions, quirk Q5; LogWeights:
    log_softmax) and the rotation matrix as _orthogonal_without_sync evaluates it.  The raw parameters are not autograd
    inputs: backward hands the whole vector-Jacobian product, the rotation's included, to the optimiser's flat gradient."""

    @staticmethod
    def forward(ctx, opt, pack, anchor):
        raw = opt.flat.detach()
        w = torch.empty_like(raw)
        L.check(L.load().pmt_constraints_forward(raw.data_ptr(), pack.mask.data_ptr(), raw.numel(), pack.table.data_ptr(),
                                                 pack.n_groups, w.data_ptr(), torch.cuda.current_stream(raw.device).cuda_stream))
        if pack.rotation is not None:
            _, module, attr, off, n = pack.rotation
            w[off:off + n] = _orthogonal_without_sync(module, attr).reshape(-1)
        ctx.opt, ctx.pack = opt, pack
        ctx.save_for_backward(raw, w)
        return w

    @staticmethod
    def backward(ctx, d_flat):
        opt, pack = ctx.opt, ctx.pack
        raw, w = ctx.saved_tensors
        lib, stream = L.load(), torch.cuda.current_stream(d_flat.device).cuda_stream
        d_flat = d_flat.contiguous()
        g = torch.empty_like(d_flat)
        L.check(lib.pmt_constraints_backward(raw.data_ptr(), w.data_ptr(), d_flat.data_ptr(), pack.mask.data_ptr(), d_flat.numel(),
                                             pack.table.data_ptr(), pack.n_groups, g.data_ptr(), stream))
        if pack.rotation is not None and pack.rotation[0].requires_grad:
            X, module, attr, off, n = pack.rotation
            dQ = d_flat[off:off + n]
            if X.shape[0] <= _ROTATION_KERNEL_MAX_N:          # _RotationFunction.backward, written into the slot
                base = getattr(getattr(module.parametrizations, attr)[0], "base", None)
                base = None if base is None else base.detach().contiguous()
                L.check(lib.pmt_orthogonal_backward(raw[off:off + n].data_ptr(), None if base is None else base.data_ptr(),
                                                    dQ.data_ptr(), X.shape[0], g[off:off + n].data_ptr(), stream))
            else:
                with torch.enable_grad():
                    dX, = torch.autograd.grad(_orthogonal_without_sync(module, attr), X, dQ.view(X.shape))
                g[off:off + n] = dX.reshape(-1)
        opt.receive_flat_gradient(g)
        return None, None, None


def materialize_flat(opt) -> torch.Tensor:
    """The training-time path of ``ArtifactModel.flat_weights`` when a FlatAdamW backs the parameters."""
    pack = opt._constraint_pack
    return _FastMaterialize.apply(opt, pack, pack.anchor)


def _mlp_ops(offsets: Dict[str, int], prefix: str, layer_sizes: List[int]):
    """mlp.py:39-66 as a flat program of Linear ops."""
    ops, idx, in_dim = [], 0, layer_sizes[0]
    n_entries = len(layer_sizes) - 1
    for k, width in enumerate(layer_sizes[1:]):
        if width < 0:
            depth = -width
            for j in range(depth):
                flags = (L.OP_SKIP_BEGIN if j == 0 else 0) | (L.OP_SKIP_END if j == depth - 1 else L.OP_POST_SELU)
                base = f"{prefix}._model.{idx}.mlp._model.{2 * j + 1}"
                ops.append(L.PmtLinearOp(in_dim, in_dim, offsets[base + ".weight"], offsets[base + ".bias"],
                                         offsets[f"{prefix}._model.{idx}.alpha"], flags))
            idx += 1
            continue
        post = k < n_entries - 1
        base = f"{prefix}._model.{idx}"
        ops.append(L.PmtLinearOp(in_dim, width, offsets[base + ".weight"], offsets[base + ".bias"], -1,
                                 L.OP_POST_SELU if post else 0))
        idx += 2 if post else 1
        in_dim = width
    if len(ops) > L.MAX_MLP_OPS:
        raise NotImplementedError(f"{prefix}: more than {L.MAX_MLP_OPS} linear layers")
    return ops


def _cnn_ops(offsets: Dict[str, int], prefix: str, layers: List[dict]):
    """dna_sequence_convolution.py:57-99 as conv / pool / linear ops with activations folded into the
    preceding conv or linear (a monotone activation commutes exactly with the max-pools between)."""
    ops = []
    act_code = {"selu": L.ACT_SELU, "leaky_relu": L.ACT_LEAKY_RELU}
    for i, rec in enumerate(layers):
        kind = rec["kind"]
        if kind == "convolution":
            ops.append(L.PmtCnnOp(L.CNN_CONV, rec["in_ch"], rec["out_ch"], rec["kernel_size"], 1, rec["in_len"],
                                  rec["out_len"], L.ACT_NONE, offsets[f"{prefix}._model.{i}.weight"],
                                  offsets[f"{prefix}._model.{i}.bias"]))
        elif kind == "pool":
            ops.append(L.PmtCnnOp(L.CNN_POOL, rec["in_ch"], rec["in_ch"], rec["kernel_size"],
                                  rec.get("stride", rec["kernel_size"]), rec["in_len"], rec["out_len"], L.ACT_NONE, -1, -1))
        elif kind in act_code:
            target = next((o for o in reversed(ops) if o.kind in (L.CNN_CONV, L.CNN_LINEAR)), None)
            if target is None or target.act != L.ACT_NONE:
                raise NotImplementedError("activation without a preceding conv/linear layer, or two in a row")
            target.act = act_code[kind]
        elif kind == "flatten":
            continue
        elif kind == "linear":
            ops.append(L.PmtCnnOp(L.CNN_LINEAR, rec["in_ch"], rec["out_ch"], 1, 1, 1, 1, L.ACT_NONE,
                                  offsets[f"{prefix}._model.{i}.weight"], offsets[f"{prefix}._model.{i}.bias"]))
    if len(ops) > L.MAX_CNN_OPS:
        raise NotImplementedError(f"haplotype CNN: more than {L.MAX_CNN_OPS} layers")
    return ops


def build_desc(model, read_row_bytes: int = 12) -> L.PmtModelDesc:
    offsets, n_params = flat_layout(model)
    hp = model._params
    d = L.PmtModelDesc()
    d.abi_version = L.PMT_ABI_VERSION
    d.n_read_features = model.read_embedding.input_dimension()
    d.read_row_bytes = d.n_read_features - 56 + 7
    d.n_info_features = model.info_embedding.input_dimension()
    d.hap_len = model.haplotypes_length() // 2
    d.d_read = model.read_embedding.output_dimension()
    d.d_info = model.info_embedding.output_dimension()
    d.d_seq = model.haplotypes_cnn.output_dimension()
    d.d_model = d.d_read + d.d_info + d.d_seq
    d.d_ffn = hp.self_attention_hidden_dimension
    d.n_blocks = hp.num_self_attention_layers
    d.d_feat = model.reducer.output_dimension()
    d.n_clusters = hp.num_artifact_clusters
    if d.n_blocks > L.MAX_BLOCKS:
        raise NotImplementedError(f"more than {L.MAX_BLOCKS} gated blocks")

    for field, count, ops in (
            ("read_ops", "n_read_ops", _mlp_ops(offsets, "read_embedding", [d.n_read_features] + list(hp.read_layers))),
            ("info_ops", "n_info_ops", _mlp_ops(offsets, "info_embedding", [d.n_info_features] + list(hp.info_layers))),
            ("red_ops", "n_red_ops", _mlp_ops(offsets, "reducer", [d.d_model] + list(hp.aggregation_layers))),
            ("cnn_ops", "n_cnn_ops", _cnn_ops(offsets, "haplotypes_cnn", model.haplotypes_cnn.layers))):
        setattr(d, count, len(ops))
        arr = getattr(d, field)
        for i, op in enumerate(ops):
            arr[i] = op

    for b in range(d.n_blocks):
        p = f"ref_alt_reads_encoder.blocks.{b}"
        o = d.blocks[b]
        o.ln_w, o.ln_b = offsets[p + ".norm.weight"], offsets[p + ".norm.bias"]
        o.p1_ref_w, o.p1_ref_b = offsets[p + ".proj1_ref.weight"], offsets[p + ".proj1_ref.bias"]
        o.p1_alt_w, o.p1_alt_b = offsets[p + ".proj1_alt.weight"], offsets[p + ".proj1_alt.bias"]
        o.alpha_ref, o.alpha_alt = offsets[p + ".sgu.alpha_ref"], offsets[p + ".sgu.alpha_alt"]
        o.beta_ref, o.beta_alt = offsets[p + ".sgu.beta_ref"], offsets[p + ".sgu.beta_alt"]
        o.gamma = offsets[p + ".sgu.gamma"]
        o.regularizer = offsets[p + ".sgu.ref_regularizer"]
        o.ln2_w, o.ln2_b = offsets[p + ".sgu.norm.weight"], offsets[p + ".sgu.norm.bias"]
        o.reg_weight = offsets[p + ".sgu.parametrizations.reg_weight.original"]
        o.p2_ref_w, o.p2_ref_b = offsets[p + ".proj2_ref.weight"], offsets[p + ".proj2_ref.bias"]
        o.p2_alt_w, o.p2_alt_b = offsets[p + ".proj2_alt.weight"], offsets[p + ".proj2_alt.bias"]

    d.translation = offsets["pre_clustering_transform.translation_e"]
    d.rotation = offsets["pre_clustering_transform.rotation_ee.parametrizations.weight.original"]
    fc = "feature_clustering"
    d.sigma_e = offsets[fc + ".parametrizations.nonartifact_stdev_e.original"]
    d.unit_ke = offsets[fc + ".parametrizations.artifact_directions_ke.original"]
    d.tau_k = offsets[fc + ".parametrizations.artifact_stdev_k.original"]
    d.logw_k = offsets[fc + ".parametrizations.log_cluster_weights_k.original"]
    d.mu_k = offsets[fc + ".artifact_emg.mu_k"]
    d.emg_sigma_k = offsets[fc + ".artifact_emg.parametrizations.sigma_k.original"]
    d.lambda_k = offsets[fc + ".artifact_emg.parametrizations.lambda_k.original"]
    d.n_params = n_params
    return d


def build_loss_desc(model, max_outlier_logit: float, max_alt_count: float) -> L.PmtLossDesc:
    """Kernel-facing description of the loss head (artifact_model.py:267-279, 299-325): the two adversarial MLP
    programs with offsets into the same flat weight buffer as build_desc."""
    offsets, n_params = flat_layout(model)
    d = L.PmtLossDesc()
    d.d_feat = model.reducer.output_dimension()
    d.n_sources = model.num_sources
    alt = _mlp_ops(offsets, "alt_count_predictor.wrapped_module", model.alt_count_predictor.wrapped_module.layer_sizes)
    src = [] if model.num_sources == 1 else _mlp_ops(offsets, "source_predictor.wrapped_module",
                                                     model.source_predictor.wrapped_module.layer_sizes)
    for ops in (alt, src):
        for op in ops:
            if max(op.in_dim, op.out_dim) > L.MAX_HEAD_DIM:
                raise NotImplementedError(f"adversarial head layers wider than {L.MAX_HEAD_DIM} are not supported")
    d.n_alt_ops, d.n_src_ops = len(alt), len(src)
    for i, op in enumerate(alt):
        d.alt_ops[i] = op
    for i, op in enumerate(src):
        d.src_ops[i] = op
    d.alt_reversal = float(model.alt_count_predictor.gradient_reversal.alpha)
    d.src_reversal = float(model.source_predictor.gradient_reversal.alpha)
    d.max_outlier_logit, d.max_alt_count = float(max_outlier_logit), float(max_alt_count)
    d.n_params = n_params
    return d
