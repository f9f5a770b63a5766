"""Times the posterior-model fit of many samples side by side on synthetic posterior records (bench.run_posterior's
generator, as profiles/time_posterior_fit.py uses it; each sample its own slice of records) at batch 64:

1. one pass of pmt_posterior_fit_pass_many over N samples for several N (CUDA events, mean of 3 passes after a warm-up
   pass), beside N x one pmt_posterior_fit_pass on a single sample timed the same way;
2. the host M step per model (update_priors_m_step, host clock with a synchronise), first half of the iterations
   (context-dependent SNV priors off) and second half (on: the float64 context fit on the CPU);
3. a whole learn_priors_and_spectra_together against each model's own learn_priors_and_spectra, one after the other
   (host clock), and whether both give the same histories and state dicts.

Prints the card, its power limit and the host's usable CPUs from the same run.
python profiles/time_posterior_fit_many.py [records_per_sample] [N,N,...] [e2e_N] [e2e_iterations] [together_only_N]"""
import copy
import ctypes as C
import os
import subprocess
import sys
import time

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R, os.path.join(R, "profiles")]
import torch  # noqa: E402


def _timed_passes(launch, passes, dev):
    launch()                                       # warm-up
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    ev0.record()
    for _ in range(passes):
        launch()
    ev1.record()
    torch.cuda.synchronize(dev)
    return ev0.elapsed_time(ev1) / passes


def main():
    from time_posterior_fit import synthetic_records
    from permutect_b200.architecture.posterior_model import (PosteriorModel, PosteriorRecords, _DeviceFit, _usable_cpus,
                                                            learn_priors_and_spectra_together)
    from permutect_b200.engine import library as L
    per = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000
    ns = [int(x) for x in sys.argv[2].split(",")] if len(sys.argv) > 2 else [1, 16, 148, 296]
    e2e_n = int(sys.argv[3]) if len(sys.argv) > 3 else 16
    e2e_iterations = int(sys.argv[4]) if len(sys.argv) > 4 else 10
    together_only_n = int(sys.argv[5]) if len(sys.argv) > 5 else 148
    passes = 3
    dev = torch.device("cuda:0")
    print("card, power limit:", subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                               capture_output=True, text=True).stdout.strip())
    print(f"SMs: {torch.cuda.get_device_properties(dev).multi_processor_count}, usable host CPUs: {_usable_cpus()}, "
          f"torch threads: {torch.get_num_threads()}")
    n_max = max(ns + [e2e_n, together_only_n])
    it, ft = synthetic_records(n_max * per, dev)
    records = [PosteriorRecords(it[i * per:(i + 1) * per], ft[i * per:(i + 1) * per], batch_size=64, device=dev) for i in range(n_max)]
    lib = L.load()
    stream = torch.cuda.current_stream(dev).cuda_stream

    # ---- 1. one pass ----
    fits = []
    for r in records:
        m = PosteriorModel(-10.0, -10.0, device=dev)
        f = _DeviceFit(m, r, 0.001)
        fits.append((f, f.begin_pass(1, 2)))       # first half: context-dependent SNV priors off
    p0 = fits[0][1]
    ws1 = torch.empty(int(lib.pmt_posterior_fit_pass_workspace_size(5)), dtype=torch.uint8, device=dev)

    def single():
        L.check(lib.pmt_posterior_fit_pass(C.byref(p0.desc), p0.params, p0.raw_params, p0.adam_m, p0.adam_v, p0.adam_step, p0.learning_rate,
                                           p0.int_array, p0.int_stride, p0.float_array, p0.float_kind, p0.float_stride, p0.n_records,
                                           p0.batch_size, p0.batch_losses_out, p0.posterior_totals_tc, p0.somatic_snv_totals_rrra,
                                           p0.snv_context_totals_rrra, ws1.data_ptr(), ws1.numel(), stream))

    t1 = _timed_passes(single, passes, dev)
    print(f"single sample (pmt_posterior_fit_pass): {per} records, {len(records[0])} batches of 64: {t1:.1f} ms per pass")
    print("| samples N | one pmt_posterior_fit_pass_many pass | N x single-sample pass | ratio to one single pass |")
    print("|---|---|---|---|")
    for n in ns:
        arr = (L.PmtPosteriorFitProblem * n)(*[p for _, p in fits[:n]])
        ws = torch.empty(int(lib.pmt_posterior_fit_pass_many_workspace_size(n, 5)), dtype=torch.uint8, device=dev)
        tn = _timed_passes(lambda: L.check(lib.pmt_posterior_fit_pass_many(arr, n, ws.data_ptr(), ws.numel(), stream)), passes, dev)
        assert all(bool(torch.isfinite(f.losses).all()) for f, _ in fits[:n])
        print(f"| {n} | {tn:.1f} ms | {n * t1:.1f} ms | {tn / t1:.2f} |")

    # ---- 2. host M step per model ----
    n_m = min(16, n_max)
    for f, _ in fits[:n_m]:
        f.end_pass()
    for label, context in (("first half (context priors off)", False), ("second half (context priors on)", True)):
        if context:                                # the first context fit of a process loads torch's optimiser code
            f = fits[0][0]
            f.model.priors.enable_context_dependent_snv_priors()
            t0 = time.perf_counter()
            f.model.update_priors_m_step(f.totals_tc, 10.0, f.somatic_snv_rrra, f.snv_context_rrra)
            print(f"host M step, first context fit of the process: {1e3 * (time.perf_counter() - t0):.0f} ms")
        times = []
        for f, _ in fits[:n_m]:
            if context:
                f.model.priors.enable_context_dependent_snv_priors()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            f.model.update_priors_m_step(f.totals_tc, 10.0, f.somatic_snv_rrra, f.snv_context_rrra)
            torch.cuda.synchronize(dev)
            times.append(time.perf_counter() - t0)
        print(f"host M step per model, {label}: mean {1e3 * sum(times) / len(times):.1f} ms, min {1e3 * min(times):.1f}, "
              f"max {1e3 * max(times):.1f} over {n_m} models; {n_m} in sequence {1e3 * sum(times):.0f} ms")
    del fits

    # ---- 3. end to end ----
    def fresh(n):
        return [PosteriorModel(-10.0, -10.0, device=dev) for _ in range(n)]

    models = fresh(e2e_n)
    alone = [copy.deepcopy(m) for m in models]
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    want = [m.learn_priors_and_spectra(r, e2e_iterations, 10.0) for m, r in zip(alone, records)]
    torch.cuda.synchronize(dev)
    t_seq = time.perf_counter() - t0
    t0 = time.perf_counter()
    got = learn_priors_and_spectra_together(models, records[:e2e_n], e2e_iterations, 10.0)
    torch.cuda.synchronize(dev)
    t_tog = time.perf_counter() - t0
    same = got == want and all(all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), s.state_dict().values()))
                               for m, s in zip(models, alone))
    print(f"{e2e_iterations} iterations, {e2e_n} samples of {per} records: learn_priors_and_spectra one model after another "
          f"{t_seq:.1f} s, learn_priors_and_spectra_together {t_tog:.1f} s ({t_seq / t_tog:.1f}x); "
          f"histories and state dicts bitwise equal: {same}")
    if together_only_n:
        models = fresh(together_only_n)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        learn_priors_and_spectra_together(models, records[:together_only_n], e2e_iterations, 10.0)
        torch.cuda.synchronize(dev)
        print(f"{e2e_iterations} iterations, {together_only_n} samples of {per} records: learn_priors_and_spectra_together "
              f"{time.perf_counter() - t0:.1f} s")


if __name__ == "__main__":
    main()
