"""CUDA-graph replay of the hot path at the batch sizes the reference's tools actually use (64 variants by default:
parameters.py:214, tools/filter_variants.py:81).  At those sizes the step is bound by the host (ctypes, autograd over the
parametrised tensors, ~60 launches), not by the kernels; every kernel of the path is free of host synchronisation and takes
its exact sizes from device memory, so a whole call -- or a whole optimisation step -- is captured once and replayed.

    infer = GraphedInference(model, example_batch)            # filter_variants.py:292-320, one batch per call
    out = infer(batch)                                         # BatchOutput over persistent tensors (valid until the next call)

    step = GraphedTrainStep(model, optimizer, example_batch)   # model_training.py:151-165 for one (downsampled) batch
    loss = step(batch)                                         # forward + losses + backward + all-reduce + clip + AdamW

A batch is replayed when it has the captured number of variants, fits the captured row capacity and holds no read set
longer than a tile; anything else takes the eager path (same results).  Capturing bakes in what the host passed by value:
the learning rate (re-captured when it changes), the precision mode, the set of trainable tensors.
"""
from typing import Optional

import torch

from permutect_b200.data.batch import Batch
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L

MAX_TILE_SET = 125      # a set of up to PMT_TILE_ROWS - 3 rows always fits one tile (pmt_host.h)


def _static_batch(example: Batch, device, row_capacity: int, index_capacity: Optional[int]) -> Batch:
    """A Batch over persistent device buffers of fixed capacity with the example's column layout."""
    b = Batch.__new__(Batch)
    b.int_tensor = torch.zeros((example.size(), example.int_tensor.shape[1]), dtype=example.int_tensor.dtype, device=device)
    b.float_tensor = torch.zeros((example.size(), example.float_tensor.shape[1]), dtype=example.float_tensor.dtype, device=device)
    b.reads_are_compressed = example.reads_are_compressed
    b.reads = torch.zeros((row_capacity,) + tuple(example.reads.shape[1:]), dtype=example.reads.dtype, device=device)
    b.max_rows_per_variant = MAX_TILE_SET
    b.read_indices = None if index_capacity is None else torch.zeros(index_capacity, dtype=torch.int64, device=device)
    b._dataset_order = False
    b._finish_initialization_from_arrays()
    if index_capacity is not None:
        b._device_counts = (torch.zeros(example.size(), dtype=torch.int64, device=device),
                            torch.ones(example.size(), dtype=torch.int64, device=device))
    return b


def _fits(static: Batch, batch: Batch) -> bool:
    if batch.size() != static.size() or batch.max_rows_per_variant > MAX_TILE_SET or getattr(batch, "_dataset_order", False):
        return False
    if batch.reads.shape[0] > static.reads.shape[0] or (batch.read_indices is None) != (static.read_indices is None):
        return False
    return batch.read_indices is None or batch.read_indices.shape[0] <= static.read_indices.shape[0]


def _load(static: Batch, batch: Batch):
    """Copies a batch into the persistent buffers (asynchronous; pinned host or device sources)."""
    static.int_tensor.copy_(batch.int_tensor, non_blocking=True)
    static.float_tensor.copy_(batch.float_tensor, non_blocking=True)
    static.reads[:batch.reads.shape[0]].copy_(batch.reads, non_blocking=True)
    if static.read_indices is not None:
        static.read_indices[:batch.read_indices.shape[0]].copy_(batch.read_indices, non_blocking=True)
        ref_counts, alt_counts = batch.counts()
        static._device_counts[0].copy_(ref_counts, non_blocking=True)
        static._device_counts[1].copy_(alt_counts, non_blocking=True)


def _capture(fn, device, warmup: int = 3):
    """Warm-up calls on a side stream (lazy initialisation, and for inference the call that packs the weight images into
    the private workspace: the later calls -- and so the capture -- take pmt_forward_prepared), then the capture."""
    stream = torch.cuda.Stream(device)
    stream.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(stream):
        for _ in range(warmup):
            fn()
    torch.cuda.current_stream(device).wait_stream(stream)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        result = fn()
    return graph, result


class GraphedInference:
    def __init__(self, model, example: Batch, row_capacity: Optional[int] = None):
        self.model, self.device = model, model._device
        rows = row_capacity or max(int(example.reads.shape[0] * 1.5) + 64, 64 * example.size())
        self.static = _static_batch(example, self.device, rows, None)
        _load(self.static, example)
        self.workspace = None
        self._key = None
        self._capture()

    def _capture(self):
        desc = self.model.descriptor()
        need = L.load().pmt_workspace_size(engine.C.byref(desc), engine.C.byref(self.static.pmt_batch()), 0)
        if self.workspace is None or self.workspace.numel() < need:
            self.workspace = torch.empty(int(need) + 4096, dtype=torch.uint8, device=self.device)
        self.static._offsets = None

        def call():
            self.static._offsets = None          # the offsets are recomputed from the persistent counts inside the graph
            with torch.inference_mode():
                return self.model.compute_batch_output(self.static)

        self._flat = self.model.flat_weights()
        self._key = (L.get_precision(), self._flat.data_ptr(), self._flat._version if not self._flat.is_inference() else None)
        with engine.use_workspace(self.device, self.workspace):
            self.graph, self.output = _capture(call, self.device)

    def __call__(self, batch: Batch):
        if not _fits(self.static, batch):
            with torch.inference_mode():
                return self.model.compute_batch_output(batch if batch.reads.device == self.device else batch.copy_to(self.device))
        flat = self.model.flat_weights()
        key = (L.get_precision(), flat.data_ptr(), flat._version if not flat.is_inference() else None)
        if key != self._key:                     # the weights (or the arithmetic mode) changed since the capture
            self._capture()
        _load(self.static, batch)
        self.graph.replay()
        return self.output


class GraphedTrainStep:
    """One optimisation step of model_training.py:151-165 (compute_batch_output, compute_batch_losses,
    misc_utils.backpropagate) for a batch -- typically a DownsampledBatch built eagerly, whose keep decisions need a fresh
    seed every step -- replayed from a CUDA graph.  Returns the summed loss (a persistent device scalar)."""

    def __init__(self, model, optimizer, example: Batch, process_group=None, row_capacity: Optional[int] = None):
        from permutect_b200.training.step import backpropagate
        self.model, self.optimizer, self.device, self.process_group = model, optimizer, model._device, process_group
        self._backpropagate = backpropagate
        rows = row_capacity or max(int(example.reads.shape[0] * 1.5) + 64, 64 * example.size())
        idx = None if example.read_indices is None else rows
        self.static = _static_batch(example, self.device, rows, idx)
        if idx is not None and example.read_indices.shape[0] > idx:
            raise ValueError("row capacity smaller than the example batch")
        _load(self.static, example)
        self.workspace = None
        self._capture()

    def _capture(self):
        lib, desc = L.load(), self.model.descriptor()
        pb = self.static.pmt_batch()
        need = max(lib.pmt_workspace_size(engine.C.byref(desc), engine.C.byref(pb), 0),
                   lib.pmt_workspace_size(engine.C.byref(desc), engine.C.byref(pb), 1),
                   lib.pmt_head_backward_workspace_size(engine.C.byref(desc)))
        if self.workspace is None or self.workspace.numel() < need:
            self.workspace = torch.empty(int(need) + 4096, dtype=torch.uint8, device=self.device)
        # the optimiser state must not move during the warm-up replays of the capture
        saved = [t.clone() for t in (self.optimizer.flat, self.optimizer.exp_avg, self.optimizer.exp_avg_sq, self.optimizer.step_count)]
        saved_step = self.optimizer._step

        def call():
            self.static._offsets = None
            with engine.use_workspace(self.device, self.workspace):
                output = self.model.compute_batch_output(self.static)
                losses = self.model.compute_batch_losses(output, self.static)
                self._backpropagate(self.optimizer, losses.total_loss, params_to_clip=self.model.parameters(),
                                    process_group=self.process_group)
            return losses.total_loss.detach()

        self._key = (L.get_precision(), float(self.optimizer.param_groups[0]["lr"]),
                     tuple(p.requires_grad for p in self.model.parameters()))
        self.graph, self.loss = _capture(call, self.device)
        with torch.no_grad():
            for t, s in zip((self.optimizer.flat, self.optimizer.exp_avg, self.optimizer.exp_avg_sq, self.optimizer.step_count), saved):
                t.copy_(s)
        self.optimizer._step = saved_step

    def __call__(self, batch: Batch):
        key = (L.get_precision(), float(self.optimizer.param_groups[0]["lr"]), tuple(p.requires_grad for p in self.model.parameters()))
        if not _fits(self.static, batch):
            from permutect_b200.training.step import train_step
            _, losses = train_step(self.model, batch, self.optimizer, process_group=self.process_group)
            return losses.total_loss.detach()
        if key != self._key:
            self._capture()
        _load(self.static, batch)
        self.graph.replay()
        self.optimizer._step += 1
        return self.loss
