"""ctypes binding of libpermutect_b200.so (C-ABI declared in include/permutect_b200.h).

The structures below mirror the header field for field.  The library is located in-tree
(``permutect_b200/csrc/libpermutect_b200.so``, built by ``permutect_b200.csrc.build``); if it is
missing the compute entry points raise -- there is no fallback implementation.
"""
import ctypes as C
import os

PMT_ABI_VERSION = 4
MAX_MLP_OPS, MAX_BLOCKS, MAX_CNN_OPS = 16, 12, 16
MAX_DIM, MAX_INFO_DIM, MAX_FEAT, MAX_CLUSTERS, TILE_ROWS = 64, 128, 32, 14, 128

OP_POST_SELU, OP_SKIP_BEGIN, OP_SKIP_END = 1, 2, 4
CNN_CONV, CNN_POOL, CNN_LINEAR = 1, 2, 3
ACT_NONE, ACT_SELU, ACT_LEAKY_RELU = 0, 1, 2
READS_U8, READS_F32, READS_F16 = 0, 1, 2
F32, F16 = 0, 1
I16, I64 = 0, 1

PRECISION_MODES = {"fp32": 0, "tf32x3": 1, "tf32": 2}

_i32 = C.c_int32


class PmtLinearOp(C.Structure):
    _fields_ = [("in_dim", _i32), ("out_dim", _i32), ("w_off", _i32), ("b_off", _i32), ("alpha_off", _i32),
                ("flags", _i32)]


class PmtCnnOp(C.Structure):
    _fields_ = [("kind", _i32), ("in_ch", _i32), ("out_ch", _i32), ("ksize", _i32), ("stride", _i32),
                ("in_len", _i32), ("out_len", _i32), ("act", _i32), ("w_off", _i32), ("b_off", _i32)]


class PmtBlockOffsets(C.Structure):
    _fields_ = [(n, _i32) for n in (
        "ln_w", "ln_b", "p1_ref_w", "p1_ref_b", "p1_alt_w", "p1_alt_b", "alpha_ref", "alpha_alt", "beta_ref",
        "beta_alt", "gamma", "regularizer", "ln2_w", "ln2_b", "reg_weight", "p2_ref_w", "p2_ref_b", "p2_alt_w",
        "p2_alt_b")]


class PmtModelDesc(C.Structure):
    _fields_ = ([(n, _i32) for n in (
        "abi_version", "n_read_features", "read_row_bytes", "n_info_features", "hap_len", "d_read", "d_info", "d_seq",
        "d_model", "d_ffn", "n_blocks", "d_feat", "n_clusters", "n_read_ops", "n_info_ops", "n_red_ops", "n_cnn_ops")]
        + [("read_ops", PmtLinearOp * MAX_MLP_OPS), ("info_ops", PmtLinearOp * MAX_MLP_OPS),
           ("red_ops", PmtLinearOp * MAX_MLP_OPS), ("cnn_ops", PmtCnnOp * MAX_CNN_OPS),
           ("blocks", PmtBlockOffsets * MAX_BLOCKS)]
        + [(n, _i32) for n in ("translation", "rotation", "sigma_e", "unit_ke", "tau_k", "logw_k", "mu_k",
                               "emg_sigma_k", "lambda_k", "n_params")])


class PmtBatch(C.Structure):
    _fields_ = [("n_variants", _i32), ("reads_kind", _i32), ("info_kind", _i32), ("hap_kind", _i32),
                ("n_rows", C.c_int64), ("total_ref", C.c_int64), ("max_rows_per_variant", C.c_int64),
                ("reads", C.c_void_p), ("read_indices", C.c_void_p), ("ref_off", C.c_void_p), ("alt_off", C.c_void_p),
                ("info", C.c_void_p), ("info_stride", C.c_int64), ("haplotypes", C.c_void_p), ("hap_stride", C.c_int64)]


class PmtOutputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("logits_bk", "logits_b", "outlier_logits_b", "alt_means_be", "ref_means_be",
                                          "info_seq_be", "final_re")]


class PmtOutGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("d_logits_bk", "d_alt_means_be", "d_ref_means_be", "info_seq_be", "saved")]


MAX_HEAD_DIM = 32


class PmtLossDesc(C.Structure):
    _fields_ = [("d_feat", _i32), ("n_sources", _i32), ("n_alt_ops", _i32), ("n_src_ops", _i32),
                ("alt_ops", PmtLinearOp * MAX_MLP_OPS), ("src_ops", PmtLinearOp * MAX_MLP_OPS),
                ("alt_reversal", C.c_float), ("src_reversal", C.c_float), ("max_outlier_logit", C.c_float),
                ("max_alt_count", C.c_float), ("n_params", _i32)]


class PmtLossBatch(C.Structure):
    _fields_ = [("n_variants", _i32), ("label_col", _i32), ("source_col", _i32), ("alt_count_col", _i32),
                ("int_array", C.c_void_p), ("int_stride", C.c_int64), ("alt_counts", C.c_void_p),
                ("logits_b", C.c_void_p), ("outlier_logits_b", C.c_void_p), ("features_be", C.c_void_p),
                ("weights_b", C.c_void_p), ("source_weights_b", C.c_void_p)]


class PmtLossOutputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("supervised_b", "unsupervised_b", "alt_count_b", "source_b", "total_b")]


class PmtLossGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("g_supervised_b", "g_unsupervised_b", "g_alt_count_b", "g_source_b", "g_total_b")]


EXPORTED_SYMBOLS = ["pmt_posterior_fit_step", "pmt_posterior_fit_workspace_size", "pmt_posterior_fit_pass",
                    "pmt_posterior_fit_pass_workspace_size", "pmt_posterior_fit_pass_many", "pmt_posterior_fit_pass_many_workspace_size",
                    "pmt_posterior_fit_ctas", "pmt_orthogonal_forward", "pmt_orthogonal_backward", "pmt_posterior_param_count", "pmt_posterior_log_posteriors", "pmt_dataset_read_indices", "pmt_pack_posterior", "pmt_adamw_step", "pmt_adamw_workspace_size", "pmt_losses_forward", "pmt_losses_backward", "pmt_losses_workspace_size", "pmt_last_error", "pmt_abi_version", "pmt_workspace_size", "pmt_forward", "pmt_forward_prepared", "pmt_backward",
                    "pmt_decode_reads", "pmt_set_profile_events", "pmt_downsample_counts", "pmt_downsample_fill", "pmt_set_precision", "pmt_get_precision", "pmt_constraints_forward", "pmt_constraints_backward", "pmt_backward_kernels", "pmt_train_saved_bytes", "pmt_forward_train",
                    "pmt_head_backward_workspace_size", "pmt_head_backward", "pmt_snv_context_fit_many", "pmt_snv_context_fit_workspace_size"]

class PmtPosteriorDesc(C.Structure):
    _fields_ = [("n_components", C.c_int32), ("hap_start", C.c_int32), ("hap_len", C.c_int32), ("no_germline_mode", C.c_int32),
                ("use_context_dependent_snv_priors", C.c_int32), ("het_beta", C.c_float)]


class PmtPosteriorFitProblem(C.Structure):
    _fields_ = [("desc", PmtPosteriorDesc), ("params", C.c_void_p), ("raw_params", C.c_void_p), ("adam_m", C.c_void_p),
                ("adam_v", C.c_void_p), ("adam_step", C.c_void_p), ("learning_rate", C.c_double), ("int_array", C.c_void_p),
                ("int_stride", C.c_int64), ("float_array", C.c_void_p), ("float_kind", C.c_int32), ("float_stride", C.c_int64),
                ("n_records", C.c_int64), ("batch_size", C.c_int32), ("batch_losses_out", C.c_void_p),
                ("posterior_totals_tc", C.c_void_p), ("somatic_snv_totals_rrra", C.c_void_p), ("snv_context_totals_rrra", C.c_void_p)]


class PmtPosteriorOutputs(C.Structure):
    _fields_ = [("log_priors_bc", C.c_void_p), ("spectra_log_lks_bc", C.c_void_p), ("normal_log_lks_bc", C.c_void_p),
                ("log_posteriors_bc", C.c_void_p), ("posterior_probabilities_bc", C.c_void_p)]


class PmtConstraintGroup(C.Structure):
    _fields_ = [("type", C.c_int32), ("off", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32), ("a", C.c_float), ("b", C.c_float)]


CONSTRAINT_EXP, CONSTRAINT_BOUNDED, CONSTRAINT_UNIT, CONSTRAINT_UNIT_TWICE, CONSTRAINT_LOGSOFTMAX = 0, 1, 2, 3, 4

_LIB = None


def library_path() -> str:
    override = os.environ.get("PERMUTECT_B200_LIBRARY")     # a differently built libpermutect_b200.so (A/B measurements)
    if override:
        return override
    return os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "csrc", "libpermutect_b200.so")


def load():
    """Load the shared library (once) and declare the prototypes of include/permutect_b200.h."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is not built; run `python -m permutect_b200.csrc.build` "
                           "(there is no CPU fallback for the ArtifactModel hot path)")
    lib = C.CDLL(path)
    lib.pmt_last_error.restype = C.c_char_p
    lib.pmt_abi_version.restype = C.c_int
    lib.pmt_workspace_size.restype = C.c_size_t
    lib.pmt_workspace_size.argtypes = [C.POINTER(PmtModelDesc), C.POINTER(PmtBatch), C.c_int]
    lib.pmt_forward.restype = C.c_int
    lib.pmt_forward.argtypes = [C.POINTER(PmtModelDesc), C.c_void_p, C.POINTER(PmtBatch), C.POINTER(PmtOutputs),
                                C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pmt_forward_prepared.restype = C.c_int
    lib.pmt_forward_prepared.argtypes = lib.pmt_forward.argtypes
    lib.pmt_train_saved_bytes.restype = C.c_size_t
    lib.pmt_train_saved_bytes.argtypes = [C.POINTER(PmtModelDesc), C.POINTER(PmtBatch)]
    lib.pmt_forward_train.restype = C.c_int
    lib.pmt_forward_train.argtypes = [C.POINTER(PmtModelDesc), C.c_void_p, C.POINTER(PmtBatch), C.POINTER(PmtOutputs),
                                      C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pmt_backward.restype = C.c_int
    lib.pmt_backward.argtypes = [C.POINTER(PmtModelDesc), C.c_void_p, C.POINTER(PmtBatch), C.POINTER(PmtOutGrads),
                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pmt_head_backward_workspace_size.restype = C.c_size_t
    lib.pmt_head_backward_workspace_size.argtypes = [C.POINTER(PmtModelDesc)]
    lib.pmt_head_backward.restype = C.c_int
    lib.pmt_head_backward.argtypes = [C.POINTER(PmtModelDesc), C.c_void_p, C.POINTER(PmtBatch), C.c_void_p,
                                      C.POINTER(PmtOutGrads), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pmt_decode_reads.restype = C.c_int
    lib.pmt_decode_reads.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
    lib.pmt_downsample_counts.restype = C.c_int
    lib.pmt_downsample_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_uint64, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pmt_downsample_fill.restype = C.c_int
    lib.pmt_downsample_fill.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_uint64, C.c_int32,
                                        C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.pmt_set_precision.restype = C.c_int
    lib.pmt_set_precision.argtypes = [C.c_int]
    lib.pmt_get_precision.restype = C.c_int
    lib.pmt_backward_kernels.restype = C.c_int
    lib.pmt_backward_kernels.argtypes = [C.POINTER(PmtModelDesc), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.pmt_set_profile_events.restype = C.c_int
    lib.pmt_set_profile_events.argtypes = [C.c_void_p, C.c_void_p]
    lib.pmt_dataset_read_indices.restype = C.c_int
    lib.pmt_dataset_read_indices.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.pmt_pack_posterior.restype = C.c_int
    lib.pmt_pack_posterior.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                       C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pmt_orthogonal_forward.restype = C.c_int
    lib.pmt_orthogonal_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.pmt_orthogonal_backward.restype = C.c_int
    lib.pmt_orthogonal_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.pmt_constraints_forward.restype = C.c_int
    lib.pmt_constraints_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.pmt_constraints_backward.restype = C.c_int
    lib.pmt_constraints_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32,
                                             C.c_void_p, C.c_void_p]
    lib.pmt_posterior_fit_workspace_size.restype = C.c_size_t
    lib.pmt_posterior_fit_workspace_size.argtypes = [C.c_int32, C.c_int32]
    lib.pmt_posterior_fit_step.restype = C.c_int
    lib.pmt_posterior_fit_step.argtypes = [C.POINTER(PmtPosteriorDesc), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int64,
                                           C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                           C.c_void_p]
    lib.pmt_posterior_fit_pass_workspace_size.restype = C.c_size_t
    lib.pmt_posterior_fit_pass_workspace_size.argtypes = [C.c_int32]
    lib.pmt_posterior_fit_pass.restype = C.c_int
    lib.pmt_posterior_fit_pass.argtypes = [C.POINTER(PmtPosteriorDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_double, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_int32,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pmt_posterior_fit_pass_many_workspace_size.restype = C.c_size_t
    lib.pmt_posterior_fit_pass_many_workspace_size.argtypes = [C.c_int32, C.c_int32]
    lib.pmt_posterior_fit_pass_many.restype = C.c_int
    lib.pmt_posterior_fit_pass_many.argtypes = [C.POINTER(PmtPosteriorFitProblem), C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pmt_posterior_fit_ctas.restype = C.c_int
    lib.pmt_posterior_fit_ctas.argtypes = [C.POINTER(PmtPosteriorFitProblem), C.c_int32]
    lib.pmt_snv_context_fit_workspace_size.restype = C.c_size_t
    lib.pmt_snv_context_fit_workspace_size.argtypes = [C.c_int32]
    lib.pmt_snv_context_fit_many.restype = C.c_int
    lib.pmt_snv_context_fit_many.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pmt_posterior_param_count.restype = C.c_int
    lib.pmt_posterior_param_count.argtypes = [C.c_int32]
    lib.pmt_posterior_log_posteriors.restype = C.c_int
    lib.pmt_posterior_log_posteriors.argtypes = [C.POINTER(PmtPosteriorDesc), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32,
                                                 C.c_int64, C.c_int32, C.POINTER(PmtPosteriorOutputs), C.c_void_p]
    lib.pmt_adamw_workspace_size.restype = C.c_size_t
    lib.pmt_adamw_step.restype = C.c_int
    lib.pmt_adamw_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                   C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t,
                                   C.c_void_p]
    lib.pmt_losses_forward.restype = C.c_int
    lib.pmt_losses_forward.argtypes = [C.POINTER(PmtLossDesc), C.c_void_p, C.POINTER(PmtLossBatch), C.POINTER(PmtLossOutputs),
                                       C.c_void_p]
    lib.pmt_losses_workspace_size.restype = C.c_size_t
    lib.pmt_losses_workspace_size.argtypes = [C.POINTER(PmtLossDesc), C.c_int32]
    lib.pmt_losses_backward.restype = C.c_int
    lib.pmt_losses_backward.argtypes = [C.POINTER(PmtLossDesc), C.c_void_p, C.POINTER(PmtLossBatch), C.POINTER(PmtLossGrads),
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    if lib.pmt_abi_version() != PMT_ABI_VERSION:
        raise RuntimeError(f"libpermutect_b200 ABI {lib.pmt_abi_version()} != binding {PMT_ABI_VERSION}")
    _LIB = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise RuntimeError("libpermutect_b200: " + load().pmt_last_error().decode())


def set_precision(mode: str) -> None:
    """Arithmetic of the read path's dense layers: "fp32" (FP32 FMA pipe, forward + backward), "tf32x3" (tcgen05
    tensor cores with split-precision TF32: the fp32-parity mode on tensor cores) or "tf32" (plain TF32 on tensor
    cores; tolerance stated separately).  In both tensor-core modes the backward runs on the tensor cores too where the
    model allows it (backward_kernels)."""
    check(load().pmt_set_precision(PRECISION_MODES[mode]))


def get_precision() -> str:
    code = load().pmt_get_precision()
    return {v: k for k, v in PRECISION_MODES.items()}[code]


def posterior_fit_ctas(problems) -> int:
    """The CTAs per problem (cluster width) with which pmt_posterior_fit_pass_many runs these PmtPosteriorFitProblem
    values, or pmt_posterior_fit_pass runs a single one (pmt_posterior_fit_ctas)."""
    arr = (PmtPosteriorFitProblem * max(len(problems), 1))(*problems)
    ctas = load().pmt_posterior_fit_ctas(arr, len(problems))
    if ctas == 0:
        raise RuntimeError("libpermutect_b200: " + load().pmt_last_error().decode())
    return ctas


def backward_kernels(desc) -> dict:
    """Which backward kernels the current precision mode runs for this model (pmt_backward_kernels)."""
    reads, cnn = C.c_int32(0), C.c_int32(0)
    check(load().pmt_backward_kernels(C.byref(desc), C.byref(reads), C.byref(cnn)))
    return {"reads_tc": bool(reads.value), "cnn_tc": bool(cnn.value)}
