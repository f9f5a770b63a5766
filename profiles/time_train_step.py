"""Times the training step and the backward kernel (CUDA events; the numbers of profiles/r1_backward_session4.md):
python profiles/time_train_step.py [n_variants] [steps]     (NOFLAT=1: per-parameter autograd path)
Prints a SHA-256 of the flat gradient of the first step, so two builds of the library compare in one line."""
import hashlib, os, sys
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R, os.path.join(R, "tests")]
import torch
import bench
from permutect_b200.data.batch import Batch, DownsampledBatch
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.synthetic import make_wgs_arrays
from permutect_b200.training.step import make_optimizer, backpropagate
from permutect_b200.utils.enums import Epoch

n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
dev = torch.device("cuda:0")
model = bench.make_model(dev); model.set_epoch_type(Epoch.TRAIN)
L.set_precision("tf32x3")
opt = make_optimizer(model)
if os.environ.get('NOFLAT'): model._flat_optimizer = None
parent = Batch.from_arrays(*make_wgs_arrays(n, seed=3000)).copy_to(dev)
g = torch.Generator().manual_seed(7)
rf, af = (0.3 + 0.7 * torch.rand(n, generator=g)).to(dev), (0.3 + 0.7 * torch.rand(n, generator=g)).to(dev)
prof = engine.ProfileEvents(dev)
def step(i, profile=False):
    b = DownsampledBatch(parent, rf, af, seed=1000 + i)
    out = model.compute_batch_output(b)
    losses = model.compute_batch_losses(out, b)
    if profile: prof.arm()
    backpropagate(opt, losses.total_loss, params_to_clip=model.parameters())
    if profile: prof.disarm()
    return losses
traj = []
for i in range(3):
    traj.append(float(step(i).total_loss.detach())/n)
    if i == 0:   # the gradients of the first step, before the optimiser has changed any weight they depend on
        g = opt.flat_grad if hasattr(opt, "flat_grad") else torch.cat([p.grad.reshape(-1) for p in model.parameters() if p.grad is not None])
        print("grad_sha256", hashlib.sha256(g.detach().float().cpu().numpy().tobytes()).hexdigest()[:16])
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(steps):
    losses = step(3 + i, True)
    traj.append(float(losses.total_loss.detach())/n)
e1.record(); torch.cuda.synchronize()
print("traj", " ".join(f"{x:.4f}" for x in traj))
print(f"tag={os.environ.get('TAG','')} n={n} step_ms={e0.elapsed_time(e1)/steps:.3f} backward_kernel_ms={prof.mean_ms():.3f} loss={float(losses.total_loss)/n:.5f}")
