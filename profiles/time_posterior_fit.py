"""Times one pass of PosteriorModel.learn_priors_and_spectra's batch loop two ways on 1.25 M synthetic posterior records
(bench.run_posterior's generator, seed 9) at batch 64: pmt_posterior_fit_pass (one launch per pass; CUDA events over
several passes after a warm-up pass) and the per-batch loop it replaces (pmt_posterior_fit_step, autograd, torch.optim.Adam;
host clock with a synchronise on both sides over a prefix of batches, reported per batch).  Prints the card and its
power limit from the same run.
python profiles/time_posterior_fit.py [n_records] [passes] [loop_batches]"""
import os, subprocess, sys, time
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R]
import torch


def synthetic_records(n, dev):
    """bench.run_posterior's posterior records: int16 [n, 58], fp32 [n, 16]."""
    g = torch.Generator(device=dev).manual_seed(9)
    it = torch.zeros((n, 16 + 42), dtype=torch.int16, device=dev)
    depth = torch.randint(8, 300, (n,), generator=g, device=dev)
    it[:, 3] = torch.randint(0, 5, (n,), generator=g, device=dev)
    it[:, 5] = depth
    it[:, 6] = torch.clamp((depth * torch.rand(n, generator=g, device=dev) * 0.6).long(), min=1)
    it[:, 7] = torch.randint(0, 200, (n,), generator=g, device=dev)
    it[:, 8] = (it[:, 7].float() * 0.03 * torch.rand(n, generator=g, device=dev)).long()
    it[:, 16:] = torch.randint(0, 4, (n, 42), generator=g, device=dev)
    ft = torch.zeros((n, 16), dtype=torch.float32, device=dev)
    ft[:, 0] = -30 * torch.rand(n, generator=g, device=dev)
    ft[:, 1] = -5 * torch.rand(n, generator=g, device=dev)
    ft[:, 2] = 10 ** (-4 * torch.rand(n, generator=g, device=dev) - 0.3)
    ft[:, 3] = 0.05 + 0.45 * torch.rand(n, generator=g, device=dev)
    ft[:, 4] = 0.05 + 0.45 * torch.rand(n, generator=g, device=dev)
    ft[:, 5] = 8 * torch.randn(n, generator=g, device=dev)
    return it, ft


def main():
    from permutect_b200.architecture.posterior_model import PosteriorModel, PosteriorRecords
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_250_000
    passes = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    loop_batches = int(sys.argv[3]) if len(sys.argv) > 3 else 2000
    dev = torch.device("cuda:0")
    print("card, power limit:", subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                               capture_output=True, text=True).stdout.strip())
    it, ft = synthetic_records(n, dev)
    records = PosteriorRecords(it, ft, batch_size=64, device=dev)

    # fused: pmt_posterior_fit_pass alone, the spectra and Adam state carried from pass to pass
    import ctypes as C
    from permutect_b200.engine import library as L
    lib = L.load()
    model = PosteriorModel(-10.0, -10.0, device=dev)
    model.priors.disable_context_dependent_snv_priors()
    raw = torch.cat([t.detach().reshape(-1) for t in model._raw_spectra_tensors()]).float().contiguous()
    m, v, step = torch.zeros_like(raw), torch.zeros_like(raw), torch.zeros(1, dtype=torch.int64, device=dev)
    ws = torch.empty(int(lib.pmt_posterior_fit_pass_workspace_size(5)), dtype=torch.uint8, device=dev)
    losses = torch.empty(len(records), device=dev)
    tc, snv, ctx = torch.zeros((5, 5), device=dev), torch.zeros((5, 5, 5, 5), device=dev), torch.zeros((5, 5, 5, 5), device=dev)
    _, _, desc, flat = model._inputs(records)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def fused_pass():
        L.check(lib.pmt_posterior_fit_pass(C.byref(desc), flat.data_ptr(), raw.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(),
                                           0.001, it.data_ptr(), it.stride(0), ft.data_ptr(), L.F32, ft.stride(0), n, 64, losses.data_ptr(),
                                           tc.data_ptr(), snv.data_ptr(), ctx.data_ptr(), ws.data_ptr(), ws.numel(), stream))

    fused_pass()                                   # warm-up
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(passes):
        fused_pass()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / passes
    assert bool(torch.isfinite(losses).all())
    print(f"fused pass (pmt_posterior_fit_pass, CUDA events, mean of {passes}): {n} records, {len(records)} batches of 64: "
          f"{ms:.1f} ms per pass, {1e3 * ms / len(records):.2f} us per batch, {n / (ms / 1e3) / 1e6:.1f} M records/s")

    # the per-batch loop on a prefix
    prefix = PosteriorRecords(it[:loop_batches * 64], ft[:loop_batches * 64], batch_size=64, device=dev)
    batches = list(prefix)
    loop = PosteriorModel(-10.0, -10.0, device=dev)
    loop.learn_priors_and_spectra(batches[:50], num_iterations=1, ignored_to_non_ignored_ratio=10.0)   # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    loop.learn_priors_and_spectra(batches, num_iterations=1, ignored_to_non_ignored_ratio=10.0)
    torch.cuda.synchronize()
    per_batch = (time.perf_counter() - t0) / len(batches)
    print(f"per-batch loop (pmt_posterior_fit_step + autograd + torch.optim.Adam): {len(batches)} batches of 64: "
          f"{1e6 * per_batch:.1f} us per batch, {per_batch * len(records):.1f} s per pass of {len(records)} batches")
    print(f"fused pass vs loop, per batch: {1e6 * per_batch / (1e3 * ms / len(records)):.1f}x")


if __name__ == "__main__":
    main()
