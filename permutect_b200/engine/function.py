"""Calls into libpermutect_b200 (C-ABI) with torch-owned device memory, and the autograd bridge.

PyTorch is plumbing here: it owns the buffers, the stream and the autograd tape that chains the
parameter-constraint Jacobians; every per-read / per-variant FLOP is executed by the library.
"""
import ctypes as C
import os
from typing import Dict, Optional

import torch

from permutect_b200.engine import library as L

_WORKSPACES: Dict[torch.device, torch.Tensor] = {}
# device -> (workspace base, weights key, precision mode) of the packed weight images currently held by the workspace
_PREPARED: Dict[torch.device, tuple] = {}


_WS_OVERRIDE: Dict[torch.device, torch.Tensor] = {}


class use_workspace:
    """Route the library calls of this device to a caller-owned workspace (engine/graphs.py: a captured CUDA graph must keep
    writing to the memory it was captured with, whatever later eager calls do to the shared workspace)."""

    def __init__(self, device: torch.device, tensor: torch.Tensor):
        self.device, self.tensor = torch.device(device), tensor

    def __enter__(self):
        self.prev = _WS_OVERRIDE.get(self.device)
        _WS_OVERRIDE[self.device] = self.tensor
        _PREPARED[self.device] = None
        return self

    def __exit__(self, *exc):
        if self.prev is None:
            _WS_OVERRIDE.pop(self.device, None)
        else:
            _WS_OVERRIDE[self.device] = self.prev
        _PREPARED[self.device] = None


def _workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    own = _WS_OVERRIDE.get(device)
    if own is not None:
        if own.numel() < nbytes:
            raise RuntimeError(f"private workspace too small: {own.numel()} < {nbytes}")
        return own
    ws = _WORKSPACES.get(device)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8, device=device)
        _WORKSPACES[device] = ws
    return ws


def _require_cuda(t: torch.Tensor):
    if t.device.type != "cuda":
        raise RuntimeError("permutect_b200 computes on CUDA devices only (no CPU fallback)")


def _check_read_width(desc: L.PmtModelDesc, batch):
    """The batch's read rows must have the model's width: the C-ABI carries no row width, so the kernels would read rows of
    any other width at the model's stride."""
    reads = batch.reads
    if reads.dtype == torch.uint8:
        want, unit = desc.read_row_bytes, "bytes (compressed)"
    else:
        want, unit = desc.n_read_features, "features (decoded)"
    if reads.dim() != 2 or reads.shape[1] != want:
        raise ValueError(f"read rows of shape {tuple(reads.shape)} do not match the model: it takes rows of {want} {unit}")


def forward_call(desc: L.PmtModelDesc, flat: torch.Tensor, batch, want_final: bool = False,
                 n_rows: Optional[int] = None, weights_key=None, for_training: bool = False) -> Dict[str, torch.Tensor]:
    """pmt_forward: one fused pass over a batch.  Returns logits_bk, logits_b, outlier_logits, alt/ref means,
    info_seq (and per-read final features when asked).

    ``weights_key``: an object that is identical (``is``) from call to call exactly as long as the contents of ``flat``
    are unchanged (the model passes the version tuple of its cached inference weights).  Consecutive calls with the
    same key, workspace and precision mode go through pmt_forward_prepared, which reuses the packed weight images.

    ``for_training``: when the library has a saved-forward path for this call (tf32x3 mode, shapes inside the tensor-core
    envelopes, buffer within its budget) the pass goes through pmt_forward_train and ``out["saved"]`` holds what the
    backward would otherwise recompute; hand it to ``backward_call``.  PERMUTECT_B200_TRAIN_SAVED=0 keeps the recompute."""
    _check_read_width(desc, batch)
    lib = L.load()
    _require_cuda(flat)
    dev = flat.device
    B, K, E = batch.size(), desc.n_clusters, desc.d_feat
    pb = batch.pmt_batch()
    f32 = dict(dtype=torch.float32, device=dev)
    out = {
        "logits_bk": torch.empty((B, K + 2), **f32), "logits_b": torch.empty(B, **f32),
        "outlier_logits": torch.empty(B, **f32), "alt_means": torch.empty((B, E), **f32),
        "ref_means": torch.empty((B, E), **f32), "info_seq": torch.empty((B, desc.d_info + desc.d_seq), **f32),
    }
    po = L.PmtOutputs(out["logits_bk"].data_ptr(), out["logits_b"].data_ptr(), out["outlier_logits"].data_ptr(),
                      out["alt_means"].data_ptr(), out["ref_means"].data_ptr(), out["info_seq"].data_ptr(), None)
    if want_final:
        out["final_re"] = torch.empty((n_rows, E), **f32)
        po.final_re = out["final_re"].data_ptr()
    need = lib.pmt_workspace_size(C.byref(desc), C.byref(pb), 0)
    if need == 0:
        raise RuntimeError("libpermutect_b200: " + lib.pmt_last_error().decode())
    ws = _workspace(dev, need)
    flat = flat.contiguous()
    state = (ws.data_ptr(), weights_key, lib.pmt_get_precision(), id(desc))
    prepared = weights_key is not None and _PREPARED.get(dev) is not None and all(
        a is b if i == 1 else a == b for i, (a, b) in enumerate(zip(_PREPARED[dev], state)))
    call = lib.pmt_forward_prepared if prepared else lib.pmt_forward
    _PREPARED[dev] = None
    saved_bytes = 0
    if for_training and os.environ.get("PERMUTECT_B200_TRAIN_SAVED", "1") != "0":
        saved_bytes = int(lib.pmt_train_saved_bytes(C.byref(desc), C.byref(pb)))
    if saved_bytes > 0:
        out["saved"] = torch.empty(saved_bytes + 256, dtype=torch.uint8, device=dev)
        base = (out["saved"].data_ptr() + 255) & ~255
        L.check(lib.pmt_forward_train(C.byref(desc), flat.data_ptr(), C.byref(pb), C.byref(po), ws.data_ptr(), ws.numel(),
                                      base, saved_bytes, torch.cuda.current_stream(dev).cuda_stream))
        return out
    L.check(call(C.byref(desc), flat.data_ptr(), C.byref(pb), C.byref(po), ws.data_ptr(), ws.numel(),
                 torch.cuda.current_stream(dev).cuda_stream))
    if weights_key is not None:
        _PREPARED[dev] = state
    return out


def backward_call(desc: L.PmtModelDesc, flat: torch.Tensor, batch, d_logits_bk: Optional[torch.Tensor],
                  d_alt_means: Optional[torch.Tensor], d_ref_means: Optional[torch.Tensor],
                  info_seq: Optional[torch.Tensor] = None, saved: Optional[torch.Tensor] = None) -> torch.Tensor:
    """pmt_backward: gradient of the fused pass w.r.t. the flat materialised weights."""
    _check_read_width(desc, batch)
    lib = L.load()
    _require_cuda(flat)
    dev = flat.device
    pb = batch.pmt_batch()
    ptr = lambda t: None if t is None else t.contiguous().data_ptr()
    keep = [None if t is None else t.contiguous() for t in (d_logits_bk, d_alt_means, d_ref_means)]
    pg = L.PmtOutGrads(*[None if t is None else t.data_ptr() for t in keep], None if info_seq is None else info_seq.data_ptr(),
                       None if saved is None else (saved.data_ptr() + 255) & ~255)
    d_flat = torch.empty_like(flat)
    need = lib.pmt_workspace_size(C.byref(desc), C.byref(pb), 1)
    if need == 0:
        raise RuntimeError("libpermutect_b200: " + lib.pmt_last_error().decode())
    ws = _workspace(dev, need)
    _PREPARED[dev] = None          # the backward rebuilds its own images in the same workspace
    L.check(lib.pmt_backward(C.byref(desc), flat.contiguous().data_ptr(), C.byref(pb), C.byref(pg), d_flat.data_ptr(),
                             ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream))
    return d_flat


def head_backward_call(desc: L.PmtModelDesc, flat: torch.Tensor, batch, final_re: torch.Tensor,
                       d_logits_bk: Optional[torch.Tensor], d_alt_means: Optional[torch.Tensor],
                       d_ref_means: Optional[torch.Tensor]) -> torch.Tensor:
    """pmt_head_backward: gradient w.r.t. the flat materialised weights of the rotation, translation and clustering
    head only (zeros elsewhere), from the per-read final features ``final_re`` of the forward of the same batch."""
    _check_read_width(desc, batch)
    lib = L.load()
    _require_cuda(flat)
    dev = flat.device
    pb = batch.pmt_batch()
    keep = [None if t is None else t.contiguous() for t in (d_logits_bk, d_alt_means, d_ref_means)]
    pg = L.PmtOutGrads(*[None if t is None else t.data_ptr() for t in keep], None, None)
    d_flat = torch.empty_like(flat)
    need = lib.pmt_head_backward_workspace_size(C.byref(desc))
    if need == 0:
        raise RuntimeError("libpermutect_b200: " + lib.pmt_last_error().decode())
    ws = _workspace(dev, need)
    _PREPARED[dev] = None          # the partial sums go to the start of the shared workspace
    L.check(lib.pmt_head_backward(C.byref(desc), flat.contiguous().data_ptr(), C.byref(pb), final_re.data_ptr(), C.byref(pg),
                                  d_flat.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream))
    return d_flat


class FusedArtifactFunction(torch.autograd.Function):
    """(flat weights, batch) -> (logits_bk, alt_means, ref_means, logits_b, outlier_logits).

    ``head_only``: nothing upstream of the rotation trains, so the backward is pmt_head_backward over the per-read final
    features this forward keeps, instead of pmt_backward over the whole model."""

    @staticmethod
    def forward(ctx, flat, desc, batch, head_only=False):
        if head_only:
            # sized from the batch's host row bound: the device offsets are not read back
            out = forward_call(desc, flat, batch, want_final=True, n_rows=int(batch.pmt_batch().n_rows))
        else:
            # keep the forward's operands only when a backward can follow (not under no_grad, not for frozen weights)
            out = forward_call(desc, flat, batch, for_training=bool(ctx.needs_input_grad[0]))
        ctx.desc, ctx.batch, ctx.head_only = desc, batch, head_only
        ctx.save_for_backward(flat, out["logits_bk"], out["logits_b"])
        ctx.info_seq = out["info_seq"]
        ctx.final_re = out.get("final_re")
        ctx.saved = out.get("saved")            # operand panels / CNN activations of the forward (None: the backward recomputes)
        ctx.saved_mode = L.get_precision()
        return out["logits_bk"], out["alt_means"], out["ref_means"], out["logits_b"], out["outlier_logits"]

    @staticmethod
    def backward(ctx, g_bk, g_alt, g_ref, g_lb, g_out):
        flat, ll, logits_b = ctx.saved_tensors
        # fold the gradients of the two derived logits into d/d logits_bk
        # (feature_clustering.py:121-135, artifact_model.py:62-73)
        g = torch.zeros_like(ll) if g_bk is None else g_bk.clone()
        if g_lb is not None:
            d_raw = g_lb * (1.0 - torch.square(logits_b / 20.0))
            g[:, 2:] += d_raw[:, None] * torch.softmax(ll[:, 2:], dim=-1)
            g[:, 0] -= d_raw
        if g_out is not None:
            non_outlier = torch.cat((ll[:, :1], ll[:, 2:]), dim=-1)
            sm = torch.softmax(non_outlier, dim=-1)
            g[:, 1] += g_out
            g[:, 0] -= g_out * sm[:, 0]
            g[:, 2:] -= g_out[:, None] * sm[:, 1:]
        if ctx.head_only:
            return head_backward_call(ctx.desc, flat, ctx.batch, ctx.final_re, g, g_alt, g_ref), None, None, None
        saved = ctx.saved if (ctx.saved is not None and L.get_precision() == ctx.saved_mode) else None
        d_flat = backward_call(ctx.desc, flat, ctx.batch, g, g_alt, g_ref, ctx.info_seq, saved)
        ctx.saved = None                        # a second backward through the same node recomputes
        return d_flat, None, None, None


def _loss_batch(batch, logits_b, outlier, features, weights, source_weights) -> L.PmtLossBatch:
    from permutect_b200.data.datum import Data
    b = L.PmtLossBatch()
    b.n_variants = batch.size()
    b.label_col, b.source_col, b.alt_count_col = Data.LABEL.idx, Data.SOURCE.idx, Data.ALT_COUNT.idx
    b.int_array, b.int_stride = batch.int_tensor.data_ptr(), batch.int_tensor.shape[1]
    dc = batch._device_counts
    b.alt_counts = dc[1].data_ptr() if dc is not None else None
    b.logits_b, b.outlier_logits_b, b.features_be = logits_b.data_ptr(), outlier.data_ptr(), features.data_ptr()
    b.weights_b = weights.data_ptr() if weights is not None else None
    b.source_weights_b = source_weights.data_ptr() if source_weights is not None else None
    return b


class FusedLossFunction(torch.autograd.Function):
    """(flat weights, logits_b, outlier logits, features_be) -> the five per-variant loss vectors of
    compute_batch_losses (artifact_model.py:299-325); forward and backward are one kernel each (pmt_losses_*)."""

    @staticmethod
    def forward(ctx, flat, logits_b, outlier, features, weights, source_weights, ldesc, batch):
        lib = L.load()
        _require_cuda(flat)
        if batch.int_tensor.device != flat.device:
            raise RuntimeError("the loss kernels need the batch on the model's CUDA device")
        tensors = [t.detach().contiguous().float() for t in (flat, logits_b, outlier, features)]
        w = None if weights is None else weights.detach().contiguous().float()
        sw = None if source_weights is None else source_weights.detach().contiguous().float()
        B = batch.size()
        out = torch.empty((5, B), dtype=torch.float32, device=flat.device)
        po = L.PmtLossOutputs(*[out[i].data_ptr() for i in range(5)])
        pb = _loss_batch(batch, tensors[1], tensors[2], tensors[3], w, sw)
        L.check(lib.pmt_losses_forward(C.byref(ldesc), tensors[0].data_ptr(), C.byref(pb), C.byref(po),
                                       torch.cuda.current_stream(flat.device).cuda_stream))
        ctx.ldesc, ctx.batch = ldesc, batch
        ctx.save_for_backward(*tensors, *(t for t in (w, sw) if t is not None))
        ctx.has_w, ctx.has_sw = w is not None, sw is not None
        return out[0], out[1], out[2], out[3], out[4]

    @staticmethod
    def backward(ctx, g_sup, g_uns, g_alt, g_src, g_tot):
        lib = L.load()
        saved = list(ctx.saved_tensors)
        flat, logits_b, outlier, features = saved[:4]
        rest = saved[4:]
        w = rest.pop(0) if ctx.has_w else None
        sw = rest.pop(0) if ctx.has_sw else None
        dev = flat.device
        keep = [None if g is None else g.contiguous().float() for g in (g_sup, g_uns, g_alt, g_src, g_tot)]
        pg = L.PmtLossGrads(*[None if g is None else g.data_ptr() for g in keep])
        pb = _loss_batch(ctx.batch, logits_b, outlier, features, w, sw)
        B = ctx.batch.size()
        d_logits, d_outlier = torch.empty(B, dtype=torch.float32, device=dev), torch.empty(B, dtype=torch.float32, device=dev)
        d_feat, d_flat = torch.empty_like(features), torch.empty_like(flat)
        need = lib.pmt_losses_workspace_size(C.byref(ctx.ldesc), B)
        ws = _workspace(dev, need)
        _PREPARED[dev] = None          # the partial sums go to the start of the shared workspace
        L.check(lib.pmt_losses_backward(C.byref(ctx.ldesc), flat.data_ptr(), C.byref(pb), C.byref(pg), d_logits.data_ptr(),
                                        d_outlier.data_ptr(), d_feat.data_ptr(), d_flat.data_ptr(), ws.data_ptr(), ws.numel(),
                                        torch.cuda.current_stream(dev).cuda_stream))
        return d_flat, d_logits, d_outlier, d_feat, None, None, None, None


class ProfileEvents:
    """CUDA-event timing of the library's dominant kernel (pmt_set_profile_events).  ``arm()`` before a
    call gives that call a fresh event pair; ``mean_ms()`` (after a synchronize) averages the pairs."""

    def __init__(self, device):
        self.device, self.pairs = device, []

    def arm(self):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream = torch.cuda.current_stream(self.device)
        a.record(stream)      # instantiates the underlying cudaEvent_t
        b.record(stream)
        L.load().pmt_set_profile_events(a.cuda_event, b.cuda_event)
        self.pairs.append((a, b))

    def disarm(self):
        L.load().pmt_set_profile_events(None, None)

    def mean_ms(self) -> float:
        self.disarm()
        times = [a.elapsed_time(b) for a, b in self.pairs]
        return sum(times) / len(times) if times else float("nan")
