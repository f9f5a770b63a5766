"""One optimisation step, as the reference's training loop performs it
(model_training.py:151-165 with misc_utils.backpropagate :125-129): forward, losses, backward,
clip_grad_norm_(1.0), AdamW.  With a process group the flat gradient is summed across ranks before
clipping, so every rank applies the identical update (SURVEY.md §8e).

On CUDA the optimiser is ``FlatAdamW``: the model's parameters become views of one flat fp32 buffer and
clip + AdamW run as two kernel launches of libpermutect_b200 (pmt_adamw_step) with no host synchronisation;
the data-parallel exchange is ONE all-reduce of the flat gradient.
"""
import ctypes as C
from typing import Iterable, Optional

import torch
from torch import nn

from permutect_b200.engine import library as L
from permutect_b200.engine import plan as planner
from permutect_b200.training import distributed as pdist


class FlatAdamW(torch.optim.Optimizer):
    """torch.optim.AdamW semantics (decoupled weight decay, bias correction, amsgrad off) preceded by
    clip_grad_norm_(max_norm) on a flat parameter buffer.  ``param_groups[0]['lr']`` is honoured every step, so
    torch LR schedulers (ReduceLROnPlateau, model_training.py:74-76) work unchanged."""

    def __init__(self, params, lr: float = 1e-3, weight_decay: float = 0.01, betas=(0.9, 0.999), eps: float = 1e-8,
                 max_norm: float = 1.0):
        params = list(params)
        super().__init__(params, dict(lr=lr, weight_decay=weight_decay, betas=betas, eps=eps, max_norm=max_norm))
        self._params = [p for g in self.param_groups for p in g["params"]]
        if not self._params or any(not p.is_cuda or p.dtype != torch.float32 for p in self._params):
            raise RuntimeError("FlatAdamW needs fp32 CUDA parameters (there is no CPU optimiser path)")
        self._sizes = [p.numel() for p in self._params]
        with torch.no_grad():
            self.flat = torch.cat([p.detach().reshape(-1) for p in self._params])
            for p, view in zip(self._params, self.flat.split(self._sizes)):
                p.data = view.view_as(p)             # parameters become views of the flat buffer
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.step_count = torch.zeros(self.flat.numel(), dtype=torch.int32, device=self.flat.device)
        self.total_norm = torch.zeros((), dtype=torch.float32, device=self.flat.device)
        self._ws = torch.empty(int(L.load().pmt_adamw_workspace_size()), dtype=torch.uint8, device=self.flat.device)
        self._step = 0
        # flat gradient path (see attach): autograd delivers d loss / d (flat materialised weights) in ONE tensor
        self.flat_grad = torch.zeros_like(self.flat)
        self._grad_views = [v.view_as(p) for p, v in zip(self._params, self.flat_grad.split(self._sizes))]
        self._flat_grad_valid = False
        self._mask_cache = (None, None)

    # ---- flat gradient path -------------------------------------------------------------------------------
    def attach(self, model):
        """Called by make_optimizer: from now on ``model.flat_weights()`` builds the materialised weight buffer from
        ``self.flat`` directly (engine/plan.py:materialize_flat: the constraint maps of every parametrised tensor, the
        rotation matrix included, in one autograd node) and its backward writes the whole gradient into
        ``self.flat_grad`` instead of ~190 per-parameter accumulations.  The host side of a training step drops from 5.7
        to 1.8 ms."""
        self._constraint_pack = planner._ConstraintPack(model, self.flat.device)
        model._flat_optimizer = self

    def backs(self, params) -> bool:
        """True while ``params`` are exactly this optimiser's parameters and still views of its flat buffer."""
        return (len(params) == len(self._params) and all(a is b for a, b in zip(params, self._params))
                and self._params[0].data_ptr() == self.flat.data_ptr())

    def receive_flat_gradient(self, d_flat: torch.Tensor):
        """Backward hook of materialize_flat: accumulate (torch semantics: gradients add up until zero_grad) and expose
        the slices as ``.grad`` of the trainable parameters."""
        if self._flat_grad_valid:
            self.flat_grad.add_(d_flat)
        else:
            self.flat_grad.copy_(d_flat)
            self._flat_grad_valid = True
        for p, view in zip(self._params, self._grad_views):
            if p.requires_grad and p.grad is None:
                p.grad = view

    def zero_grad(self, set_to_none: bool = True):
        if set_to_none:
            self._flat_grad_valid = False
            for p in self._params:
                p.grad = None
        else:
            self.flat_grad.zero_()

    def _flat_path_gradient(self):
        """(flat gradient, mask or None) when the gradient arrived through receive_flat_gradient."""
        flags = tuple(p.requires_grad and (p.grad is not None) for p in self._params)
        if all(flags):
            return self.flat_grad, None
        if self._mask_cache[0] != flags:
            dev = self.flat.device
            self._mask_cache = (flags, torch.cat([torch.full((n,), 1.0 if f else 0.0, device=dev)
                                                  for n, f in zip(self._sizes, flags)]))
        return self.flat_grad, self._mask_cache[1].clone()

    def flat_gradient(self):
        """(flat gradient, mask or None): parameters without a gradient contribute zeros and are masked out."""
        missing = [p.grad is None for p in self._params]
        if not any(missing):
            return torch.cat([p.grad.reshape(-1) for p in self._params]), None
        dev = self.flat.device
        grads = [torch.zeros(n, device=dev) if m else p.grad.reshape(-1) for p, n, m in zip(self._params, self._sizes, missing)]
        mask = torch.cat([torch.full((n,), 0.0 if m else 1.0, device=dev) for n, m in zip(self._sizes, missing)])
        return torch.cat(grads), mask

    @torch.no_grad()
    def step(self, closure=None, process_group=None):
        assert closure is None
        grad, mask = self._flat_path_gradient() if self._flat_grad_valid else self.flat_gradient()
        if process_group is not None or pdist.is_initialized():
            if mask is None:
                torch.distributed.all_reduce(grad, op=torch.distributed.ReduceOp.SUM, group=process_group)
            else:
                # ONE collective for both: a parameter frozen on this rank only must still be updated, and the kernel only
                # tests mask != 0, so the masks are summed along with the gradients
                n = grad.numel()
                packed = torch.cat((grad, mask))
                torch.distributed.all_reduce(packed, op=torch.distributed.ReduceOp.SUM, group=process_group)
                grad, mask = packed[:n], packed[n:]
        g = self.param_groups[0]
        self._step += 1
        lib = L.load()
        L.check(lib.pmt_adamw_step(self.flat.data_ptr(), grad.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
                                   self.step_count.data_ptr(), None if mask is None else mask.data_ptr(), self.flat.numel(),
                                   float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]),
                                   float(g["weight_decay"]), float(g["max_norm"]), self.total_norm.data_ptr(), self._ws.data_ptr(),
                                   self._ws.numel(), torch.cuda.current_stream(self.flat.device).cuda_stream))
        for p in self._params:                      # the kernel wrote through the views: tell autograd / caches
            torch.autograd.graph.increment_version(p)
        return None

    def state_dict(self):
        return dict(step=self._step, step_count=self.step_count.clone(), exp_avg=self.exp_avg.clone(), exp_avg_sq=self.exp_avg_sq.clone(),
                    param_groups=[{k: v for k, v in g.items() if k != "params"} for g in self.param_groups])

    def load_state_dict(self, state):
        self._step = int(state["step"])
        self.exp_avg.copy_(state["exp_avg"])
        self.step_count.copy_(state["step_count"])
        self.exp_avg_sq.copy_(state["exp_avg_sq"])
        for g, s in zip(self.param_groups, state["param_groups"]):
            g.update(s)


def make_optimizer(model: nn.Module, learning_rate: float = 1e-3, weight_decay: float = 0.01) -> torch.optim.Optimizer:
    """AdamW as in model_training.py:68-72.  On CUDA: FlatAdamW (clip + AdamW in two launches)."""
    params = [p for p in model.parameters()]
    if len(params) > 0 and params[0].is_cuda:
        opt = FlatAdamW(params, lr=learning_rate, weight_decay=weight_decay)
        if hasattr(model, "flat_weights"):
            opt.attach(model)
        return opt
    raise RuntimeError("make_optimizer needs the model's parameters on a CUDA device (FlatAdamW; there is no CPU optimiser path)")


def backpropagate(optimizer: torch.optim.Optimizer, loss: torch.Tensor, params_to_clip: Iterable[nn.Parameter] = (),
                  process_group=None):
    """misc_utils.py:125-129 (+ the data-parallel gradient sum)."""
    optimizer.zero_grad(set_to_none=True)
    loss.backward()
    if isinstance(optimizer, FlatAdamW):
        optimizer.step(process_group=process_group)      # all-reduce, clip and AdamW on the flat buffers
        return
    params_to_clip = list(params_to_clip)
    if process_group is not None or pdist.is_initialized():
        pdist.allreduce_gradients(params_to_clip, process_group)
    nn.utils.clip_grad_norm_(params_to_clip, max_norm=1.0)
    optimizer.step()


def train_step(model, batch, optimizer, balancer=None, process_group=None):
    """compute_batch_output -> compute_batch_losses -> backpropagate.  Returns (output, losses)."""
    output = model.compute_batch_output(batch, balancer)
    losses = model.compute_batch_losses(output, batch)
    backpropagate(optimizer, losses.total_loss, params_to_clip=model.parameters(), process_group=process_group)
    return output, losses
