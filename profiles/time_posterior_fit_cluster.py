"""Times the fused posterior fit pass at the cluster width the library chooses against the one-SM pass
(PMT_POSTERIOR_CTAS=1), the two forms alternating in one process on the same problems, on synthetic posterior records
(bench.run_posterior's generator, as profiles/time_posterior_fit.py uses it):

1. one sample of 1.25 M records at batch 64 and at batch 256 (pmt_posterior_fit_pass);
2. 100 k records per sample for several sample counts N at batch 64 (pmt_posterior_fit_pass_many).

Each pass is timed on its own with CUDA events, after a warm-up pass of each form; the table gives the mean and the
range of the passes.  The records (180 B each, 225 MB for 1.25 M) do not fit in the 126 MB L2.  Prints the card, its
power limit and the widths chosen from the same run.
python profiles/time_posterior_fit_cluster.py [records] [records_per_sample] [N,N,...] [passes]"""
import ctypes as C
import os
import subprocess
import sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [R, os.path.join(R, "profiles")]
import torch  # noqa: E402

FORMS = (("chosen", None), ("one CTA", "1"))


def _set_form(value):
    if value is None:
        os.environ.pop("PMT_POSTERIOR_CTAS", None)
    else:
        os.environ["PMT_POSTERIOR_CTAS"] = value


def _alternate(launch, passes, dev):
    """ms of each pass of each form, the forms alternating pass by pass after a warm-up pass of each."""
    for _, value in FORMS:
        _set_form(value)
        launch()
    times = {name: [] for name, _ in FORMS}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(passes):
        for name, value in FORMS:
            _set_form(value)
            torch.cuda.synchronize(dev)
            ev0.record()
            launch()
            ev1.record()
            torch.cuda.synchronize(dev)
            times[name].append(ev0.elapsed_time(ev1))
    _set_form(None)
    return times


def _cell(ts):
    return f"{sum(ts) / len(ts):.1f} ms ({min(ts):.1f} – {max(ts):.1f})"


def main():
    from time_posterior_fit import synthetic_records
    from permutect_b200.architecture.posterior_model import PosteriorModel, PosteriorRecords, _DeviceFit
    from permutect_b200.engine import library as L
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_250_000
    per = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000
    ns = [int(x) for x in sys.argv[3].split(",")] if len(sys.argv) > 3 else [1, 4, 16, 37, 148]
    passes = int(sys.argv[4]) if len(sys.argv) > 4 else 3
    dev = torch.device("cuda:0")
    print("card, power limit:", subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                               capture_output=True, text=True).stdout.strip())
    print(f"SMs: {torch.cuda.get_device_properties(dev).multi_processor_count}; CUDA events, mean and range of {passes} passes "
          "per form after a warm-up pass of each, the forms alternating")
    _set_form(None)
    lib = L.load()
    stream = torch.cuda.current_stream(dev).cuda_stream

    # ---- 1. one sample ----
    it, ft = synthetic_records(n, dev)
    print("| records, batch | width chosen | chosen width | one CTA | speed-up |")
    print("|---|---|---|---|---|")
    for batch in (64, 256):
        records = PosteriorRecords(it, ft, batch_size=batch, device=dev)
        fit = _DeviceFit(PosteriorModel(-10.0, -10.0, device=dev), records, 0.001)
        p = fit.begin_pass(1, 2)                   # first half: context-dependent SNV priors off
        ws = torch.empty(int(lib.pmt_posterior_fit_pass_workspace_size(p.desc.n_components)), dtype=torch.uint8, device=dev)

        def single():
            L.check(lib.pmt_posterior_fit_pass(C.byref(p.desc), p.params, p.raw_params, p.adam_m, p.adam_v, p.adam_step, p.learning_rate,
                                               p.int_array, p.int_stride, p.float_array, p.float_kind, p.float_stride, p.n_records,
                                               p.batch_size, p.batch_losses_out, p.posterior_totals_tc, p.somatic_snv_totals_rrra,
                                               p.snv_context_totals_rrra, ws.data_ptr(), ws.numel(), stream))

        width = L.posterior_fit_ctas([p])
        t = _alternate(single, passes, dev)
        assert bool(torch.isfinite(fit.losses).all())
        a, b = sum(t["chosen"]) / passes, sum(t["one CTA"]) / passes
        print(f"| {n}, {batch} | {width} | {_cell(t['chosen'])} | {_cell(t['one CTA'])} | {b / a:.2f}x |")
        del fit, records
    del it, ft

    # ---- 2. many samples ----
    n_max = max(ns)
    it, ft = synthetic_records(n_max * per, dev)
    fits = []
    for i in range(n_max):
        r = PosteriorRecords(it[i * per:(i + 1) * per], ft[i * per:(i + 1) * per], batch_size=64, device=dev)
        f = _DeviceFit(PosteriorModel(-10.0, -10.0, device=dev), r, 0.001)
        fits.append((f, f.begin_pass(1, 2)))
    print(f"| samples N ({per} records each, batch 64) | width chosen | chosen width | one CTA | speed-up |")
    print("|---|---|---|---|---|")
    for k in ns:
        arr = (L.PmtPosteriorFitProblem * k)(*[p for _, p in fits[:k]])
        ws = torch.empty(int(lib.pmt_posterior_fit_pass_many_workspace_size(k, 5)), dtype=torch.uint8, device=dev)
        width = L.posterior_fit_ctas([p for _, p in fits[:k]])
        t = _alternate(lambda: L.check(lib.pmt_posterior_fit_pass_many(arr, k, ws.data_ptr(), ws.numel(), stream)), passes, dev)
        assert all(bool(torch.isfinite(f.losses).all()) for f, _ in fits[:k])
        a, b = sum(t["chosen"]) / passes, sum(t["one CTA"]) / passes
        print(f"| {k} | {width} | {_cell(t['chosen'])} | {_cell(t['one CTA'])} | {b / a:.2f}x |")


if __name__ == "__main__":
    main()
