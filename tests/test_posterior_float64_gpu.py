"""The posterior model's kernels against the float64 oracle (oracle/posterior_model_oracle.py with dtype=torch.float64)
at every K, model configuration, float-block type and record edge (posterior_records.py):

- pmt_posterior_log_posteriors (log_posteriors_kernel<false>): the four log tables under the row bound of
  test_posterior_model.py, now up to depth 32 767; probabilities; calls; batch sizes around the 128-thread CTA; every
  output alone; haplotype lengths 3, 21 and 40 and records inside wider buffers, through the C-ABI with the descriptor
  written by hand.
- pmt_posterior_fit_step (log_posteriors_kernel<true> + fit_reduce_kernel) through negative_log_evidence and autograd:
  loss, raw-parameter gradients and the E-step totals, first on rows of depth <= 400, then on all rows.
- pmt_posterior_fit_pass and pmt_posterior_fit_pass_many (fit_pass): two carried passes against an Adam loop run in
  float64 on float64 gradients.

K, configuration, model kind, float-block type and haplotype length are crossed pairwise, not in full.  Every check
measures first, prints its worst error next to its tolerance, then asserts.  NaN in the float block is out of scope: the
reference gives NaN there, while the kernel's fminf on maf drops a NaN maf."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch
from scipy.special import gammaln

from oracle import posterior_model_oracle as orc
from posterior_records import CONFIGS, HAP_START, edge_records, model_state

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
F64 = torch.float64
KS = (1, 2, 5, 15, 16)
CONFIG_NAMES = tuple(CONFIGS)
TABLES = ("log_priors_bc", "spectra_log_lks_bc", "normal_log_lks_bc", "log_posteriors_bc")
OUTPUTS = TABLES + ("posterior_probabilities_bc",)


def _pairwise():
    """(K, config, kind, fp16, hap_len): every pair of K and configuration once; fp16, the saturated model and the haplotype
    length spread so that each meets every K and every configuration."""
    return [(K, cfg, "saturated" if (2 * i + j) % 3 == 0 else "perturbed", (i + j) % 2 == 1, (3, 21, 40)[(i + 2 * j) % 3])
            for i, K in enumerate(KS) for j, cfg in enumerate(CONFIG_NAMES)]


CASES = _pairwise()
CASE_IDS = [f"K{K}-{cfg}-{kind}-{'fp16' if fp16 else 'fp32'}-L{L}" for K, cfg, kind, fp16, L in CASES]


def _lib():
    from permutect_b200.engine import library as L
    return L, L.load()


def _model(K, config, kind, seed):
    """(GPU PosteriorModel, state dict, no_germline, het_beta, context)"""
    from permutect_b200.architecture.posterior_model import PosteriorModel, SomaticSpectrum
    sd, no_germline, het_beta, context = model_state(K, config, kind, seed)
    model = PosteriorModel(-3.0, -4.0, no_germline_mode=no_germline, device=DEV, het_beta=het_beta)
    model.spectra.somatic_spectrum = SomaticSpectrum(K).to(DEV)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    model.priors.use_context_dependent_snv_priors = context
    return model, sd, no_germline, het_beta, context


def _desc(K, hap_len, no_germline, het_beta, context):
    L, _ = _lib()
    return L.PmtPosteriorDesc(K, HAP_START, hap_len, int(no_germline), int(context), -1.0 if het_beta is None else float(het_beta))


def _on_device(ia, fa, int_pad=0, float_pad=0):
    """The records on the GPU, each row inside a row of int_pad / float_pad more columns (garbage there): (int view,
    float view) whose row strides are the wider buffer's."""
    it = torch.full((ia.shape[0], ia.shape[1] + int_pad), 4, dtype=torch.int16, device=DEV)
    ft = torch.full((fa.shape[0], fa.shape[1] + float_pad), float("nan"), dtype=torch.from_numpy(fa).dtype, device=DEV)
    it[:, :ia.shape[1]] = torch.from_numpy(ia).to(DEV)
    ft[:, :fa.shape[1]] = torch.from_numpy(fa).to(DEV)
    return it[:, :ia.shape[1]], ft[:, :fa.shape[1]]


def _log_posteriors(desc, flat, it, ft, n=None, want=OUTPUTS):
    """pmt_posterior_log_posteriors on the first n records: {output: [n, 5] numpy} of the outputs in `want`."""
    L, lib = _lib()
    n = it.shape[0] if n is None else n
    outs = {k: torch.full((max(n, 1), 5), float("nan"), device=DEV) for k in want}
    po = L.PmtPosteriorOutputs(*[outs[k].data_ptr() if k in outs else None for k in OUTPUTS])
    L.check(lib.pmt_posterior_log_posteriors(C.byref(desc), flat.data_ptr(), it.data_ptr(), it.stride(0), ft.data_ptr(),
                                             L.F16 if ft.dtype == torch.float16 else L.F32, ft.stride(0), n, C.byref(po),
                                             torch.cuda.current_stream(DEV).cuda_stream))
    torch.cuda.synchronize(DEV)
    return {k: v[:n].cpu().numpy() for k, v in outs.items()}


def _row_bound(ia, want, fa=None):
    """test_posterior_model.py's row bound: 2e-5 relative + 2e-4 + 8 float32 ulp of lgamma(depth + 2), per entry.  With
    the float block, the GERMLINE column also gets 4 float32 ulp / af: the reference's formulas log(1 - (1 - af)^2) and
    hom_prop = 1 - het_prop cancel in float32 when af is small, and the kernel computes them as the reference does
    (measured against float64: 2.5e-3 in the log prior and 1e-2 in the germline likelihood at af = 1e-5)."""
    depth = np.maximum(ia[:, 5], ia[:, 7]).astype(np.float64)
    bound = (2e-4 + 8 * np.finfo(np.float32).eps * gammaln(depth + 2.0))[:, None] + 2e-5 * np.abs(want)
    if fa is not None:
        bound[:, 3] += 4 * np.finfo(np.float32).eps / fa[:, 2].astype(np.float64)
    return bound


@functools.lru_cache(maxsize=None)
def _tables64(K, config, kind, fp16, hap_len, n_random=500, seed=0):
    ia, fa = edge_records(n_random, hap_len, fp16, seed=seed + K)
    sd, no_germline, het_beta, context = model_state(K, config, kind, seed=K)
    out = orc.log_posterior_and_ingredients(sd, ia, fa, no_germline, het_beta, context, dtype=F64)
    return ia, fa, {k: v.numpy() for k, v in out.items()}


def _check_tables(got, ia, fa, want, what):
    worst = 0.0
    for k in TABLES:
        bound = _row_bound(ia, want[k], fa)
        ratio = np.abs(got[k].astype(np.float64) - want[k]) / bound
        worst = max(worst, float(ratio.max()))
        assert np.all(np.isfinite(got[k])), (what, k)
        i = np.unravel_index(np.argmax(ratio), ratio.shape)
        assert ratio.max() <= 1, f"{what}: {k} row {i[0]} call {i[1]}: got {got[k][i]} want {want[k][i]} (depth {ia[i[0], 5]})"
    return worst


@pytest.mark.parametrize("K,config,kind,fp16,hap_len", CASES, ids=CASE_IDS)
def test_log_posteriors_against_float64(K, config, kind, fp16, hap_len):
    """Measured on an NVIDIA B200 at a 1000 W power limit: tables at most 0.41 of the row bound, probabilities 2.1e-4
    from float64, no call differs."""
    ia, fa, want = _tables64(K, config, kind, fp16, hap_len)
    model, _, no_germline, het_beta, context = _model(K, config, kind, seed=K)
    desc, flat = _desc(K, hap_len, no_germline, het_beta, context), model.flat_parameters()
    it, ft = _on_device(ia, fa)
    got = _log_posteriors(desc, flat, it, ft)
    table_worst = _check_tables(got, ia, fa, want, "tables")
    # probabilities where the row bound is below 3e-3, calls where the top two are more than twice the bound apart
    top2 = np.sort(want["log_posteriors_bc"], axis=1)[:, -2:]
    bound = _row_bound(ia, top2[:, 1:].repeat(5, axis=1), fa).max(axis=1)
    tight = bound < 3e-3
    prob_err = float(np.abs(got["posterior_probabilities_bc"][tight] - want["posterior_probabilities_bc"][tight]).max())
    decided = top2[:, 1] - top2[:, 0] > 2 * bound
    wrong = int((got["log_posteriors_bc"].argmax(1) != want["log_posteriors_bc"].argmax(1))[decided].sum())
    print(f"{len(ia)} records ({int(tight.sum())} under 3e-3, {int(decided.sum())} decided): tables {table_worst:.3f} of the row "
          f"bound, probabilities {prob_err:.2e} (tol 3e-3), {wrong} calls differ (tol 0)")
    assert tight.sum() > len(ia) // 3 and decided.mean() > 0.9
    assert prob_err <= 3e-3 and wrong == 0
    # every output requested alone: the bits of all five together
    for k in OUTPUTS:
        alone = _log_posteriors(desc, flat, it, ft, want=(k,))[k]
        assert np.array_equal(alone, got[k]), f"{k} alone differs from {k} with the other outputs"


def test_log_posteriors_batch_sizes_around_the_cta():
    """1, 127, 128, 129 and 4 097 records (the kernel's CTA is 128 threads): each against float64, and each a prefix of
    the 4 097-record launch's bits."""
    K, config, kind, fp16, hap_len = 16, "default", "saturated", False, 21
    n_edge = len(edge_records(0, hap_len)[0])
    ia, fa, want = _tables64(K, config, kind, fp16, hap_len, n_random=4097 - n_edge, seed=100)
    assert len(ia) == 4097
    model, _, no_germline, het_beta, context = _model(K, config, kind, seed=K)
    desc, flat = _desc(K, hap_len, no_germline, het_beta, context), model.flat_parameters()
    it, ft = _on_device(ia, fa)
    full = _log_posteriors(desc, flat, it, ft)
    worst = _check_tables(full, ia, fa, want, "4097 records")
    for n in (1, 127, 128, 129):
        part = _log_posteriors(desc, flat, it, ft, n)
        for k in OUTPUTS:
            assert np.array_equal(part[k], full[k][:n]), (n, k)
    print(f"4097 records: tables at {worst:.3f} of the row bound; 1, 127, 128, 129 records: the same bits")


@pytest.mark.parametrize("K,config,hap_len,fp16,int_pad,float_pad", [
    (2, "default", 3, True, 5, 3), (16, "het_beta_small", 40, False, 1, 10), (5, "no_germline", 21, True, 7, 1),
    (15, "no_context", 3, False, 2, 2)])
def test_log_posteriors_inside_wider_buffers(K, config, hap_len, fp16, int_pad, float_pad):
    """int_stride / float_stride wider than a record, with the descriptor's hap_len written by hand: the bits of the
    compact records, and float64 within the row bound."""
    ia, fa, want = _tables64(K, config, "perturbed", fp16, hap_len, n_random=300, seed=200)
    model, _, no_germline, het_beta, context = _model(K, config, "perturbed", seed=K)
    desc, flat = _desc(K, hap_len, no_germline, het_beta, context), model.flat_parameters()
    compact = _log_posteriors(desc, flat, *_on_device(ia, fa))
    wide_it, wide_ft = _on_device(ia, fa, int_pad, float_pad)
    assert wide_it.stride(0) == ia.shape[1] + int_pad and wide_ft.stride(0) == fa.shape[1] + float_pad
    wide = _log_posteriors(desc, flat, wide_it, wide_ft)
    for k in OUTPUTS:
        assert np.array_equal(wide[k], compact[k]), k
    worst = _check_tables(wide, ia, fa, want, "wide buffer")
    print(f"hap_len {hap_len}, strides +{int_pad} / +{float_pad}: same bits as compact, tables at {worst:.3f} of the row bound")


# ---- pmt_posterior_fit_step ------------------------------------------------------------------------------------------
# Gradients and totals are measured relative to each tensor's largest entry, the loss relative to itself.  Measured on an
# NVIDIA B200 at a 1000 W power limit, worst of the 25 configurations on rows of depth <= 400: loss 3.5e-6, constrained
# gradients 9.4e-4 (the K = 1 saturated model; 2.1e-4 elsewhere), raw gradients 1.9e-4, totals 2.9e-4.
STEP_TOL = dict(loss=1e-5, grad=2e-3, totals=1e-3)
SATURATED_RAW = ("spectra.somatic_spectrum.parametrizations.cf_k.original",
                 "spectra.somatic_spectrum.parametrizations.log_weights_k.original")


@functools.lru_cache(maxsize=None)
def _step64(K, config, kind, fp16, hap_len, rows):
    """Records, then (loss, d/d constrained, d/d raw) of float64 autograd and of float32 autograd (the reference's own
    precision), and the float64 posteriors."""
    ia, fa = edge_records(400, hap_len, fp16, seed=300 + K)
    if rows == "shallow":
        keep = ia[:, 5] <= 400
        ia, fa = ia[keep], fa[keep]
    sd, no_germline, het_beta, context = model_state(K, config, kind, seed=K)
    ref = {}
    for dtype in (F64, torch.float32):
        loss, con, raw = orc.negative_log_evidence_and_grads(sd, ia, fa, no_germline, het_beta, context, dtype=dtype)
        ref[dtype] = (float(loss), {k: v.double().numpy() for k, v in con.items()}, {k: v.double().numpy() for k, v in raw.items()})
    post = orc.log_posterior_and_ingredients(sd, ia, fa, no_germline, het_beta, context, dtype=F64)["posterior_probabilities_bc"].numpy()
    return ia, fa, ref[F64], ref[torch.float32], post


def _snv_cells(ia):
    L = (ia.shape[1] - HAP_START) // 2
    c = (L - 1) // 2
    h = np.clip(ia[:, HAP_START:].astype(int), 0, 4)
    return ((h[:, c - 1] * 5 + h[:, c]) * 5 + h[:, c + 1]) * 5 + h[:, c + L]


def _scaled(got, want, names=None):
    """max over tensors of max|got - want| / max|want|"""
    return max(float(np.abs(got[n] - want[n]).max()) / max(float(np.abs(want[n]).max()), 1e-30) for n in (names or want))


def _fit_step(model, ia, fa):
    """pmt_posterior_fit_step through the C-ABI: loss, {name: d/d constrained tensor} (orc.SPECTRA_RAW's names), totals."""
    from permutect_b200.architecture.posterior_model import PosteriorBatch
    L, lib = _lib()
    it, ft, desc, flat = model._inputs(PosteriorBatch(ia, fa, DEV))
    K = desc.n_components
    loss, grads = torch.empty((), device=DEV), torch.empty(2 * K + 70, device=DEV)
    tc, snv, ctx = torch.zeros((5, 5), device=DEV), torch.zeros(625, device=DEV), torch.zeros(625, device=DEV)
    ws = torch.empty(int(lib.pmt_posterior_fit_workspace_size(it.shape[0], K)), dtype=torch.uint8, device=DEV)
    L.check(lib.pmt_posterior_fit_step(C.byref(desc), flat.data_ptr(), it.data_ptr(), it.stride(0), ft.data_ptr(),
                                       L.F16 if ft.dtype == torch.float16 else L.F32, ft.stride(0), it.shape[0], loss.data_ptr(),
                                       grads.data_ptr(), tc.data_ptr(), snv.data_ptr(), ctx.data_ptr(), ws.data_ptr(), ws.numel(),
                                       torch.cuda.current_stream(DEV).cuda_stream))
    torch.cuda.synchronize(DEV)
    g, off, con = grads.cpu().numpy().astype(np.float64), 0, {}
    for name, t in zip(orc.SPECTRA_RAW, model._spectra_tensors()):
        con[name] = g[off:off + t.numel()].reshape(t.shape)
        off += t.numel()
    return float(loss), con, tc.cpu().numpy(), snv.cpu().numpy(), ctx.cpu().numpy()


STEP_CASES = [(K, cfg, kind, fp16, (3, 21)[(i + j) % 2]) for i, K in enumerate(KS) for j, cfg in enumerate(CONFIG_NAMES)
              for (_, _, kind, fp16, _) in [CASES[i * len(CONFIG_NAMES) + j]]]


def _step_id(c):
    return f"K{c[0]}-{c[1]}-{c[2]}-{'fp16' if c[3] else 'fp32'}-L{c[4]}"


@pytest.mark.parametrize("K,config,kind,fp16,hap_len", STEP_CASES, ids=[_step_id(c) for c in STEP_CASES])
def test_fit_step_on_shallow_rows_against_float64(K, config, kind, fp16, hap_len):
    """Rows of depth <= 400.  The kernel's loss, its gradients w.r.t. the constrained spectra, the raw-parameter gradients
    that negative_log_evidence's backward leaves, and the three E-step totals: posterior totals per type and call,
    somatic SNV posterior and SNV count per context cell.  On a saturated model the raw gradients of cf_k and
    log_weights_k are left out: sigmoid at +12 and a log_softmax entry 20 above the rest lose their bits in float32
    autograd itself (the float32 oracle is 3e-2 of max away from float64 there), not in the kernel."""
    from permutect_b200.architecture.posterior_model import PosteriorBatch
    ia, fa, (want_loss, want_con, want_raw), _, post = _step64(K, config, kind, fp16, hap_len, "shallow")
    model, _, _, _, _ = _model(K, config, kind, seed=K)
    loss, con, tc, snv, ctx = _fit_step(model, ia, fa)
    model.negative_log_evidence(PosteriorBatch(ia, fa, DEV)).backward()
    got_raw = {n: p.grad.cpu().numpy().astype(np.float64) for n, p in model.named_parameters() if n in want_raw}
    raw_names = [n for n in want_raw if kind != "saturated" or n not in SATURATED_RAW]
    loss_err = abs(loss - want_loss) / abs(want_loss)
    con_err, raw_err = _scaled(con, want_con), _scaled(got_raw, want_raw, raw_names)
    want_tc = np.zeros((5, 5))
    np.add.at(want_tc, ia[:, 3].astype(int), post)
    is_snv = ia[:, 3] == 0
    want_snv, want_ctx = np.zeros(625), np.zeros(625)
    np.add.at(want_snv, _snv_cells(ia)[is_snv], post[is_snv, 0])
    np.add.at(want_ctx, _snv_cells(ia)[is_snv], 1.0)
    tot_err = max(float(np.abs(tc - want_tc).max()) / float(np.abs(want_tc).max()), float(np.abs(snv - want_snv).max()) / float(want_snv.max()))
    tol = STEP_TOL
    print(f"{len(ia)} rows: loss {loss_err:.2e} (tol {tol['loss']:.0e}), gradients {con_err:.2e} constrained, {raw_err:.2e} raw of "
          f"max (tol {tol['grad']:.0e}), totals {tot_err:.2e} of max (tol {tol['totals']:.0e})")
    assert np.array_equal(ctx, want_ctx)
    assert loss_err <= tol["loss"] and con_err <= tol["grad"] and raw_err <= tol["grad"] and tot_err <= tol["totals"]


# All rows: the gradient tolerance of each configuration, 1.5 times the kernel's error measured there on an NVIDIA B200 at
# a 1000 W power limit (rounded up), and at least the shallow rows' 2e-3.  The kernel's sums run in a fixed order, so
# these records give the same error on every run.
DEEP_GRAD_TOL = {
    "K1-default-saturated-fp32-L3": 0.24,             # measured 1.59e-01
    "K1-no_context-perturbed-fp16-L21": 0.002,        # measured 9.03e-04
    "K1-het_beta-perturbed-fp32-L3": 0.0053,          # measured 3.52e-03
    "K1-het_beta_small-saturated-fp16-L21": 0.002,    # measured 9.19e-04
    "K1-no_germline-perturbed-fp32-L3": 0.0063,       # measured 4.19e-03
    "K2-default-perturbed-fp16-L21": 0.016,           # measured 1.05e-02
    "K2-no_context-saturated-fp32-L3": 0.0042,        # measured 2.75e-03
    "K2-het_beta-perturbed-fp16-L21": 0.018,          # measured 1.20e-02
    "K2-het_beta_small-perturbed-fp32-L3": 0.0087,    # measured 5.75e-03
    "K2-no_germline-saturated-fp16-L21": 0.016,       # measured 1.03e-02
    "K5-default-perturbed-fp32-L3": 0.011,            # measured 7.33e-03
    "K5-no_context-perturbed-fp16-L21": 0.012,        # measured 7.63e-03
    "K5-het_beta-saturated-fp32-L3": 0.0097,          # measured 6.42e-03
    "K5-het_beta_small-perturbed-fp16-L21": 0.0088,   # measured 5.84e-03
    "K5-no_germline-perturbed-fp32-L3": 0.011,        # measured 6.84e-03
    "K15-default-saturated-fp16-L21": 0.0079,         # measured 5.23e-03
    "K15-no_context-perturbed-fp32-L3": 0.002,        # measured 9.09e-04
    "K15-het_beta-perturbed-fp16-L21": 0.002,         # measured 5.61e-04
    "K15-het_beta_small-saturated-fp32-L3": 0.0068,   # measured 4.50e-03
    "K15-no_germline-perturbed-fp16-L21": 0.002,      # measured 8.45e-04
    "K16-default-perturbed-fp32-L3": 0.0041,          # measured 2.71e-03
    "K16-no_context-saturated-fp16-L21": 0.046,       # measured 3.03e-02
    "K16-het_beta-perturbed-fp32-L3": 0.0041,         # measured 2.67e-03
    "K16-het_beta_small-perturbed-fp16-L21": 0.006,   # measured 3.98e-03
    "K16-no_germline-saturated-fp32-L3": 0.032,       # measured 2.08e-02
}
DEEP_TOL = dict(loss=1e-4, totals=1e-2)      # measured: loss 5.6e-5 relative, totals 5.3e-3 of max at most


@pytest.mark.parametrize("K,config,kind,fp16,hap_len", STEP_CASES, ids=[_step_id(c) for c in STEP_CASES])
def test_fit_step_on_all_rows_against_float64(K, config, kind, fp16, hap_len):
    """All rows, depths up to 32 767: the checks of the shallow test.  A deep row's log tables carry the float32
    rounding of lgamma(depth + 1) (0.03 per ulp at depth 30 000; the row bound of the module docstring), and so do its
    posteriors and its gradient terms.  The reference formula evaluated in float32 (the float32 oracle, correctly
    rounded lgamma) is about as far from float64, up to 0.17 of a tensor's max on these records; the kernel, whose
    lgammaf and digammaf are not correctly rounded, is at most 3.6 times that distance.  That is the rounding the row
    bound describes, not a cancellation beyond it.  Each configuration's gradients are held to DEEP_GRAD_TOL, set
    from the kernel's error measured there; the distance of the float32 oracle is printed beside it."""
    from permutect_b200.architecture.posterior_model import PosteriorBatch
    ia, fa, (want_loss, want_con, want_raw), (_, f32_con, f32_raw), post = _step64(K, config, kind, fp16, hap_len, "all")
    model, _, _, _, _ = _model(K, config, kind, seed=K)
    loss, con, tc, snv, ctx = _fit_step(model, ia, fa)
    model.negative_log_evidence(PosteriorBatch(ia, fa, DEV)).backward()
    got_raw = {n: p.grad.cpu().numpy().astype(np.float64) for n, p in model.named_parameters() if n in want_raw}
    raw_names = [n for n in want_raw if kind != "saturated" or n not in SATURATED_RAW]
    loss_err = abs(loss - want_loss) / abs(want_loss)
    grad_err = max(_scaled(con, want_con), _scaled(got_raw, want_raw, raw_names))
    f32_err = max(_scaled(f32_con, want_con), _scaled(f32_raw, want_raw, raw_names))
    want_tc = np.zeros((5, 5))
    np.add.at(want_tc, ia[:, 3].astype(int), post)
    is_snv = ia[:, 3] == 0
    want_snv, want_ctx = np.zeros(625), np.zeros(625)
    np.add.at(want_snv, _snv_cells(ia)[is_snv], post[is_snv, 0])
    np.add.at(want_ctx, _snv_cells(ia)[is_snv], 1.0)
    tot_err = max(float(np.abs(tc - want_tc).max()) / float(np.abs(want_tc).max()), float(np.abs(snv - want_snv).max()) / float(want_snv.max()))
    print(f"{len(ia)} rows, deepest {int(ia[:, 5].max())}: loss {loss_err:.2e} (tol {DEEP_TOL['loss']:.0e}), gradients {grad_err:.2e} "
          f"of max (float32 oracle {f32_err:.2e})", end="")
    tol = DEEP_GRAD_TOL[_step_id((K, config, kind, fp16, hap_len))]
    print(f" (tol {tol:.0e}), totals {tot_err:.2e} of max (tol {DEEP_TOL['totals']:.0e})")
    assert np.array_equal(ctx, want_ctx)
    assert loss_err <= DEEP_TOL["loss"] and grad_err <= tol and tot_err <= DEEP_TOL["totals"]


# ---- pmt_posterior_fit_pass, pmt_posterior_fit_pass_many ------------------------------------------------------------
# Of each raw tensor's largest entry after two passes, or 5x the float32 loop's distance per entry.  Measured on an NVIDIA
# B200 at a 1000 W power limit: at most 2.6e-4 of max, 0.26 of an entry's tolerance, alone and in the many-launch.
PASS_TOL = 1e-3
# Pairwise: each K and configuration meets every batch size and both rates.  Each problem's records alternate edge rows
# (some of depth 0, whose spectra gradients are zero) and random rows.  Batch 1 runs at lr 0.001 only: at lr 0.05
# its single-record gradients of the log weights, r_k - p_k for components of tiny responsibility, cancel and change
# sign from step to step, and Adam's division by their RMS turns float32 rounding into full steps (measured: 1.1e-2 of
# max at K = 16, which a second float32 implementation, the oracle, does not reproduce entry for entry).
PASS_CASES = [(K, cfg, (1, 7, 64)[(i + j) % 3], 0.001 if (i + j) % 3 == 0 or (i + j) % 2 else 0.05)
              for i, K in enumerate((1, 5, 16)) for j, cfg in enumerate(CONFIG_NAMES)]
N_RECORDS = {1: 13, 7: 40, 64: 150}      # 13 and 6 batches, and 3 with a last one of 22


def _adam_loop(sd, ia, fa, batch_size, lr, no_germline, het_beta, context, dtype):
    """The raw spectra after two passes of Adam (float64 arithmetic) on the oracle's gradients in `dtype` at the current
    raw values (rounded to `dtype`), and the number of steps."""
    names = list(orc.SPECTRA_RAW.values())
    p = {k: sd[k].astype(np.float64) for k in names}
    m = {k: np.zeros_like(p[k]) for k in names}
    v = {k: np.zeros_like(p[k]) for k in names}
    t = 0
    for _ in range(2):
        for lo in range(0, len(ia), batch_size):
            t += 1
            cur = dict(sd)
            cur.update({k: torch.from_numpy(p[k]).to(dtype) for k in names})
            _, _, g = orc.negative_log_evidence_and_grads(cur, ia[lo:lo + batch_size], fa[lo:lo + batch_size], no_germline, het_beta,
                                                         context, dtype=dtype)
            for k in names:
                gk = g[k].double().numpy()
                m[k] = 0.9 * m[k] + 0.1 * gk
                v[k] = 0.999 * v[k] + 0.001 * gk * gk
                p[k] = p[k] - lr / (1 - 0.9 ** t) * m[k] / (np.sqrt(v[k]) / np.sqrt(1 - 0.999 ** t) + 1e-8)
    return [p[k] for k in names], t


@functools.lru_cache(maxsize=None)
def _pass_problem(K, config, batch_size, lr):
    """Records (fp16, depth <= 400), the raw spectra after two passes of float64 Adam on float64 oracle gradients, the
    step count, and the per-entry tolerance of a float32 implementation: PASS_TOL of the tensor's largest entry, or 5
    times the distance of the same loop on float32 oracle gradients where that is larger.  Adam divides each gradient by
    its running RMS, so an entry whose gradient is small and changes sign from step to step carries float32 rounding
    into the parameters at full step size (measured: 0.14 of max in one artifact alpha at batch 1, lr 0.05)."""
    n = N_RECORDS[batch_size]
    ia, fa = edge_records(n, 21, True, seed=400 + K, max_depth=400)
    # edge and random rows taken in turn, so that every batch size, batch 1 too, sees both
    n_edge = len(edge_records(0, 21)[0])
    edge, rand = [i for i in range(n_edge) if ia[i, 5] <= 400], list(range(n_edge, len(ia)))
    order = [i for pair in zip(edge, rand) for i in pair] + edge[len(rand):] + rand[len(edge):]
    ia, fa = ia[order[:n]], fa[order[:n]]
    sd, no_germline, het_beta, context = model_state(K, config, "perturbed", seed=K)
    want, t = _adam_loop(sd, ia, fa, batch_size, lr, no_germline, het_beta, context, F64)
    f32, _ = _adam_loop(sd, ia, fa, batch_size, lr, no_germline, het_beta, context, torch.float32)
    tol = [np.maximum(PASS_TOL * max(float(np.abs(w).max()), 1e-30), 5 * np.abs(a - w)) for a, w in zip(f32, want)]
    return ia, fa, want, t, tol


class _Pass:
    """One fit-pass problem's arguments and its carried buffers (raw, m, v, step)."""

    def __init__(self, K, config, batch_size, lr):
        self.ia, self.fa, self.want, self.steps, self.tol = _pass_problem(K, config, batch_size, lr)
        self.model, _, no_germline, het_beta, context = _model(K, config, "perturbed", seed=K)
        self.desc = _desc(K, 21, no_germline, het_beta, context)
        self.flat = self.model.flat_parameters()
        self.it, self.ft = _on_device(self.ia, self.fa)
        self.batch_size, self.lr = batch_size, lr
        self.raw = torch.cat([t.detach().reshape(-1) for t in self.model._raw_spectra_tensors()]).float().contiguous()
        self.m, self.v = torch.zeros_like(self.raw), torch.zeros_like(self.raw)
        self.step = torch.zeros(1, dtype=torch.int64, device=DEV)
        n_batches = -(-len(self.ia) // batch_size)
        self.losses = torch.empty(n_batches, device=DEV)
        self.tc, self.snv, self.ctx = torch.zeros((5, 5), device=DEV), torch.zeros(625, device=DEV), torch.zeros(625, device=DEV)

    def next_pass(self):
        """The constrained values of the carried raw spectra, as the kernel's `params` of the next pass."""
        off = 0
        with torch.no_grad():
            for t in self.model._raw_spectra_tensors():
                t.copy_(self.raw[off:off + t.numel()].reshape(t.shape))
                off += t.numel()
        self.flat = self.model.flat_parameters()

    def struct(self):
        L, _ = _lib()
        return L.PmtPosteriorFitProblem(self.desc, self.flat.data_ptr(), self.raw.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                                        self.step.data_ptr(), self.lr, self.it.data_ptr(), self.it.stride(0), self.ft.data_ptr(),
                                        L.F16, self.ft.stride(0), len(self.ia), self.batch_size, self.losses.data_ptr(),
                                        self.tc.data_ptr(), self.snv.data_ptr(), self.ctx.data_ptr())

    def run_alone(self):
        L, lib = _lib()
        s = self.struct()
        ws = torch.empty(int(lib.pmt_posterior_fit_pass_workspace_size(s.desc.n_components)), dtype=torch.uint8, device=DEV)
        L.check(lib.pmt_posterior_fit_pass(C.byref(s.desc), s.params, s.raw_params, s.adam_m, s.adam_v, s.adam_step, s.learning_rate,
                                           s.int_array, s.int_stride, s.float_array, s.float_kind, s.float_stride, s.n_records,
                                           s.batch_size, s.batch_losses_out, s.posterior_totals_tc, s.somatic_snv_totals_rrra,
                                           s.snv_context_totals_rrra, ws.data_ptr(), ws.numel(), torch.cuda.current_stream(DEV).cuda_stream))
        torch.cuda.synchronize(DEV)

    def error(self):
        """(max over raw tensors of max|kernel - float64| / max|float64|, the largest ratio of an entry's error to its
        tolerance, the tensor where that is)"""
        got, off = self.raw.cpu().numpy().astype(np.float64), 0
        scaled, worst = 0.0, (0.0, None)
        for name, w, tol in zip(orc.SPECTRA_RAW, self.want, self.tol):
            err = np.abs(got[off:off + w.size].reshape(w.shape) - w)
            off += w.size
            scaled = max(scaled, float(err.max()) / max(float(np.abs(w).max()), 1e-30))
            worst = max(worst, (float((err / tol).max()), name))
        return (scaled,) + worst


def _run_many(problems):
    L, lib = _lib()
    arr = (L.PmtPosteriorFitProblem * len(problems))(*[p.struct() for p in problems])
    max_k = max(p.desc.n_components for p in problems)
    ws = torch.empty(int(lib.pmt_posterior_fit_pass_many_workspace_size(len(problems), max_k)), dtype=torch.uint8, device=DEV)
    L.check(lib.pmt_posterior_fit_pass_many(arr, len(problems), ws.data_ptr(), ws.numel(), torch.cuda.current_stream(DEV).cuda_stream))
    torch.cuda.synchronize(DEV)


@pytest.mark.parametrize("K,config,batch_size,lr", PASS_CASES)
def test_fit_pass_follows_float64_adam(K, config, batch_size, lr):
    """Two passes that carry raw, m, v and step (the second pass's bias corrections continue from the first's last step)."""
    p = _Pass(K, config, batch_size, lr)
    p.run_alone()
    p.next_pass()
    p.run_alone()
    err, ratio, where = p.error()
    print(f"{len(p.ia)} records, batch {batch_size}, lr {lr}: {p.steps} Adam steps, raw {err:.2e} of each tensor's max, worst entry "
          f"at {ratio:.2f} of its tolerance ({where})")
    assert int(p.step) == p.steps and bool(torch.isfinite(p.losses).all())
    assert ratio <= 1


def test_fit_pass_many_with_mixed_k_follows_float64_adam():
    """Every problem of PASS_CASES (K 1, 5 and 16) in one pmt_posterior_fit_pass_many launch per pass, two passes."""
    problems = [_Pass(*c) for c in PASS_CASES]
    _run_many(problems)
    for p in problems:
        p.next_pass()
    _run_many(problems)
    errs = [p.error()[1] for p in problems]
    print(f"{len(problems)} problems, mixed K: worst raw error at {max(errs):.2f} of its problem's tolerance")
    assert [int(p.step) for p in problems] == [p.steps for p in problems]
    assert max(errs) <= 1
