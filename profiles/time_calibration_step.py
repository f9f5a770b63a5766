"""Times a calibration step (only model.calibration_parameters() train) on the head-only backward against the same step
with one trunk tensor unfrozen (the reducer's last bias: the whole model's backward, what the step cost before the head
path existed), alternating the two in one process, and pmt_head_backward alone.  CUDA events; v0.4.0 model, tf32x3,
downsampled WGS batches, FlatAdamW.
python profiles/time_calibration_step.py [n_variants] [steps]"""
import os, subprocess, sys
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R, os.path.join(R, "tests")]
import torch
import bench
from permutect_b200.data.batch import Batch, DownsampledBatch
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.synthetic import make_wgs_arrays
from permutect_b200.training.model_training import freeze, unfreeze
from permutect_b200.training.step import make_optimizer, backpropagate
from permutect_b200.utils.enums import Epoch

n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
dev = torch.device("cuda:0")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip())
model = bench.make_model(dev)
model.set_epoch_type(Epoch.TRAIN)
L.set_precision("tf32x3")
opt = make_optimizer(model)
parent = Batch.from_arrays(*make_wgs_arrays(n, seed=3000)).copy_to(dev)
g = torch.Generator().manual_seed(7)
rf, af = (0.3 + 0.7 * torch.rand(n, generator=g)).to(dev), (0.3 + 0.7 * torch.rand(n, generator=g)).to(dev)
last_bias = [p for name, p in model.named_parameters() if name.startswith("reducer") and name.endswith("bias")][-1]


def set_path(full: bool):
    freeze(model.parameters())
    unfreeze(model.calibration_parameters())
    last_bias.requires_grad = full


def step(i):
    b = DownsampledBatch(parent, rf, af, seed=1000 + i)
    losses = model.compute_batch_losses(model.compute_batch_output(b), b)
    backpropagate(opt, losses.total_loss, params_to_clip=model.parameters())


# calibration gradients of one batch on both paths
b = DownsampledBatch(parent, rf, af, seed=999)
grads = {}
for full in (False, True):
    set_path(full)
    opt.zero_grad(set_to_none=True)
    model.compute_batch_losses(model.compute_batch_output(b), b).total_loss.backward()
    grads[full] = [p.grad.detach().clone() for p in model.calibration_parameters()]
diff = max(float((a - c).abs().max() / c.abs().max()) for a, c in zip(grads[False], grads[True]))
print(f"calibration gradients, head path vs full backward: largest difference {diff:.2e} of the tensor's max")

ms = {False: [], True: []}
for i in range(3):                       # warm-up of both paths
    for full in (False, True):
        set_path(full)
        step(i)
torch.cuda.synchronize()
for i in range(steps):
    for full in (False, True):
        set_path(full)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(10 + i)
        e1.record()
        torch.cuda.synchronize()
        ms[full].append(e0.elapsed_time(e1))

# pmt_head_backward alone, on the outputs of one head-path forward
set_path(False)
desc = model.descriptor()
with torch.no_grad():
    out = engine.forward_call(desc, model.flat_weights(), b, want_final=True, n_rows=int(b.pmt_batch().n_rows))
g_bk, g_alt, g_ref = (torch.randn_like(out[k]) for k in ("logits_bk", "alt_means", "ref_means"))
flat = model.flat_weights().detach()
for _ in range(5):
    engine.head_backward_call(desc, flat, b, out["final_re"], g_bk, g_alt, g_ref)
reps = 50
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    engine.head_backward_call(desc, flat, b, out["final_re"], g_bk, g_alt, g_ref)
e1.record()
torch.cuda.synchronize()
med = lambda xs: sorted(xs)[len(xs) // 2]
rows = int((b.counts()[0].sum() + b.counts()[1].sum()).item())
print(f"n={n} rows={rows} steps={steps} head_path_step_ms={med(ms[False]):.3f} full_backward_step_ms={med(ms[True]):.3f} "
      f"head_backward_call_ms={e0.elapsed_time(e1) / reps:.3f}  (medians; min {min(ms[False]):.3f} / {min(ms[True]):.3f})")

# device time of head_backward_kernel itself, in a profiled run of its own
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(20):
        engine.head_backward_call(desc, flat, b, out["final_re"], g_bk, g_alt, g_ref)
    torch.cuda.synchronize()
for ev in prof.key_averages():
    if "head_backward_kernel" in ev.key or "head_finish_kernel" in ev.key:
        print(f"{ev.key.split('(')[0]}: {ev.device_time_total / ev.count / 1000:.3f} ms per launch ({ev.count} launches)")
