"""Times the haplotype-CNN stage of the resident inference forward: the split pair (hap_cnn_tc_kernel over the head layers,
hap_cnn_tail_kernel) against the single kernel (PMT_CNN_SINGLE=1), alternating in one process.
    python profiles/time_cnn_forward.py [n_variants] [launches] [runs] [precision]
Per run and arm: CUDA events around `launches` prepared forward calls (the whole step), then a torch.profiler run of its
own over as many calls for each CNN kernel's device time.  PMT_CNN_SINGLE=0 keeps the pair at batches below its
batch-size threshold.  The last lines give the kernel names and a SHA-256 of
info_seq's sequence columns per arm."""
import hashlib, os, statistics, sys
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R, os.path.join(R, "tests")]
import torch
from torch.profiler import ProfilerActivity, profile
import bench
from permutect_b200.data.batch import Batch
from permutect_b200.engine import function as engine
from permutect_b200.engine import library as L
from permutect_b200.synthetic import make_wgs_arrays

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1250000
launches = int(sys.argv[2]) if len(sys.argv) > 2 else 20
runs = int(sys.argv[3]) if len(sys.argv) > 3 else 5
mode = sys.argv[4] if len(sys.argv) > 4 else "tf32x3"
dev = torch.device("cuda:0")
model = bench.make_model(dev)
L.set_precision(mode)
batch = Batch.from_arrays(*make_wgs_arrays(n, seed=3000)).copy_to(dev)
desc, flat = model.descriptor(), model.flat_weights()
KEY = object()
ARMS = {"split": "0", "single": "1"}


def call():
    return engine.forward_call(desc, flat, batch, weights_key=KEY)


def kernel_ms():
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        for _ in range(launches):
            call()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if "hap_cnn" in e.key:
            t = getattr(e, "device_time_total", None)
            out[e.key] = (t if t is not None else e.cuda_time_total) / 1e3 / launches
    return out


step, cnn, per_kernel, digest = {a: [] for a in ARMS}, {a: [] for a in ARMS}, {a: {} for a in ARMS}, {}
with torch.inference_mode():
    for r in range(runs):
        for arm, flag in ARMS.items():
            os.environ["PMT_CNN_SINGLE"] = flag
            for _ in range(3):
                out = call()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                call()
            e1.record()
            torch.cuda.synchronize()
            step[arm].append(e0.elapsed_time(e1) / launches)
            ks = kernel_ms()
            cnn[arm].append(sum(ks.values()))
            for k, v in ks.items():
                per_kernel[arm].setdefault(k, []).append(v)
            print(f"run {r} {arm}: step_ms={step[arm][-1]:.3f} cnn_ms={cnn[arm][-1]:.3f} " +
                  " ".join(f"{k.split('(')[0].split('::')[-1].replace(' ', '')}={v:.3f}" for k, v in ks.items()), flush=True)
            if r == 0:
                d_info = desc.d_info
                digest[arm] = hashlib.sha256(out["info_seq"][:, d_info:].contiguous().cpu().numpy().tobytes()).hexdigest()[:16]
os.environ.pop("PMT_CNN_SINGLE", None)
spread = lambda v: max(v) - min(v)
print(f"n={n} launches={launches} runs={runs} mode={mode}")
for arm in ARMS:
    print(f"{arm}: cnn stage median {statistics.median(cnn[arm]):.3f} ms (spread {spread(cnn[arm]):.3f}), "
          f"step median {statistics.median(step[arm]):.3f} ms (spread {spread(step[arm]):.3f})")
    for k, v in per_kernel[arm].items():
        print(f"  {statistics.median(v):.3f} ms (spread {spread(v):.3f})  {k}")
print("sha256 info_seq[:, d_info:] " + " ".join(f"{a}={h}" for a, h in digest.items()))
