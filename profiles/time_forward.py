"""Times ArtifactModel.compute_batch_output on a resident WGS-shaped shard (CUDA events) and the read kernel inside it:
python profiles/time_forward.py [n_variants] [steps] [precision]        (PMT_TC_PACKED=0: the sequential tile planner)
The last line holds a SHA-256 of every BatchOutput field, so two builds of the library compare in one line."""
import hashlib, os, sys
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R, os.path.join(R, "tests")]
import torch
import bench
from permutect_b200.data.batch import Batch
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.synthetic import make_wgs_arrays

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1250000
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
mode = sys.argv[3] if len(sys.argv) > 3 else "tf32x3"
dev = torch.device("cuda:0")
model = bench.make_model(dev)
L.set_precision(mode)
batch = Batch.from_arrays(*make_wgs_arrays(n, seed=3000)).copy_to(dev)
prof = engine.ProfileEvents(dev)
with torch.inference_mode():
    for _ in range(3):
        out = model.compute_batch_output(batch)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof.arm()
    e0.record()
    for _ in range(steps):
        out = model.compute_batch_output(batch)
    e1.record()
    torch.cuda.synchronize()
    prof.disarm()
ms = e0.elapsed_time(e1) / steps
print(f"packed={os.environ.get('PMT_TC_PACKED', '1')} n={n} step_ms={ms:.3f} read_kernel_ms={prof.mean_ms():.3f} "
      f"variants_per_s={n / ms * 1e3:.4g} checksum={float(out.logits_b.double().sum()):.6f}")
digest = {k: hashlib.sha256(v.detach().float().contiguous().cpu().numpy().tobytes()).hexdigest()[:16]
          for k, v in sorted(vars(out).items()) if isinstance(v, torch.Tensor)}
print("sha256 " + " ".join(f"{k}={h}" for k, h in digest.items()))
