"""Times the posterior model's context-dependent SNV-prior fit on the host and on the device.

1. The fits alone, for N models: the in-process host fit (fit_mutation_rates_sc, one after another), ContextFitPool over
   the host's usable CPUs (as learn_priors_and_spectra_together runs it), and one pmt_snv_context_fit_many launch
   (fit_mutation_rates_sc_on_device).  The totals come from real passes: each sample's 100 k synthetic records
   (bench.run_posterior's generator, as profiles/time_posterior_fit_many.py uses it) take one second-half pass of
   pmt_posterior_fit_pass_many, and its E-step totals are rounded as the M step rounds them.  Also prints the largest
   relative gap between the device's and the host's rates.
2. learn_priors_and_spectra_together over N samples for ten iterations, context_fit="host" against "device",
   alternating in this process.

Host clock around work that ends in a device synchronise.  Prints the card and its power limit from the same run.
python profiles/time_context_fit.py [records_per_sample] [N,N,...] [iterations] [rounds]"""
import os
import subprocess
import sys
import time

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R, os.path.join(R, "profiles")]
import torch  # noqa: E402


def _clock(fn, dev):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize(dev)
    return time.perf_counter() - t0, out


def main():
    from time_posterior_fit import synthetic_records
    from permutect_b200.architecture.posterior_model import (PosteriorModel, PosteriorRecords, _DeviceFit, _usable_cpus,
                                                            learn_priors_and_spectra_together)
    from permutect_b200.architecture.snv_context_priors import (ContextFitPool, fit_mutation_rates_sc,
                                                              fit_mutation_rates_sc_on_device)
    from permutect_b200.engine import library as L
    per = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000
    ns = [int(x) for x in sys.argv[2].split(",")] if len(sys.argv) > 2 else [1, 16, 148]
    iterations = int(sys.argv[3]) if len(sys.argv) > 3 else 10
    rounds = int(sys.argv[4]) if len(sys.argv) > 4 else 1
    dev = torch.device("cuda:0")
    print("card, power limit:", subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                               capture_output=True, text=True).stdout.strip())
    print(f"SMs: {torch.cuda.get_device_properties(dev).multi_processor_count}, usable host CPUs: {_usable_cpus()}, "
          f"torch threads: {torch.get_num_threads()}")
    n_max = max(ns)
    it, ft = synthetic_records(n_max * per, dev)
    records = [PosteriorRecords(it[i * per:(i + 1) * per], ft[i * per:(i + 1) * per], batch_size=64, device=dev) for i in range(n_max)]

    # ---- the fits' inputs from one second-half pass per sample ----
    lib = L.load()
    fits = [_DeviceFit(PosteriorModel(-10.0, -10.0, device=dev), r, 0.001) for r in records]
    problems = (L.PmtPosteriorFitProblem * n_max)(*[f.begin_pass(2, 2) for f in fits])
    ws = torch.empty(int(lib.pmt_posterior_fit_pass_many_workspace_size(n_max, 5)), dtype=torch.uint8, device=dev)
    L.check(lib.pmt_posterior_fit_pass_many(problems, n_max, ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream))
    torch.cuda.synchronize(dev)
    del ws
    inputs = []
    for f in fits:
        f.end_pass()
        inputs.append(f.model._m_step_before_context_fit(f.totals_tc, 10.0, f.somatic_snv_rrra, f.snv_context_rrra))
    total = torch.stack([t for t, _ in inputs])
    snv = torch.stack([s for _, s in inputs])
    print(f"inputs: {n_max} samples of {per} records, cell totals {float(total.min()):.3g}..{float(total.max()):.3g}, "
          f"SNVs per cell {float(snv.min()):.0f}..{float(snv.max()):.0f}")
    del fits

    # ---- 1. the fits alone ----
    fit_mutation_rates_sc(*inputs[0])                          # loads torch's optimiser code
    fit_mutation_rates_sc_on_device(inputs[:1], dev)           # loads the module, computes the draw tables
    workers = min(n_max, _usable_cpus())
    pool = ContextFitPool(workers) if workers > 1 else None
    if pool is not None:
        pool.map(inputs[:workers])
    print("| models N | host, in process | ContextFitPool | one device launch | host / device | max relative rate gap |")
    print("|---|---|---|---|---|---|")
    for n in ns:
        t_host, host = _clock(lambda: [fit_mutation_rates_sc(*x) for x in inputs[:n]], dev)
        t_pool, _ = _clock(lambda: pool.map(inputs[:n]), dev) if pool is not None and n > 1 else (float("nan"), None)
        t_dev, got = _clock(lambda: fit_mutation_rates_sc_on_device(inputs[:n], dev), dev)
        gap = max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(got, host))
        print(f"| {n} | {1e3 * t_host:.0f} ms | {1e3 * t_pool:.0f} ms | {1e3 * t_dev:.1f} ms | {t_host / t_dev:.0f}x | {gap:.1e} |")
    if pool is not None:
        pool.close()

    # ---- 2. learn_priors_and_spectra_together, host against device context fits ----
    print(f"| samples N | {iterations} iterations, context_fit=\"host\" | context_fit=\"device\" | host / device |")
    print("|---|---|---|---|")
    for n in ns:
        times = {"host": [], "device": []}
        for _ in range(rounds):
            for where in ("host", "device"):
                models = [PosteriorModel(-10.0, -10.0, device=dev) for _ in range(n)]
                t, _ = _clock(lambda: learn_priors_and_spectra_together(models, records[:n], iterations, 10.0, context_fit=where), dev)
                times[where].append(t)
        th, td = min(times["host"]), min(times["device"])
        print(f"| {n} | {th:.2f} s | {td:.2f} s | {th / td:.1f}x |")


if __name__ == "__main__":
    main()
