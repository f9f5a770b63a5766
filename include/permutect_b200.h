/*
 * permutect_b200 C-ABI: the ArtifactModel hot path on NVIDIA B200 (sm_100a).
 *
 * The reference (broadinstitute/permutect) is pure Python/PyTorch and has no FFI; the boundary it
 * exposes for this path is the Python surface of permutect/architecture/artifact_model.py
 * (ArtifactModel.compute_batch_output :281, compute_batch_losses :299, calculate_features :239).
 * Underneath that surface this library is what a maintainer would bind (ctypes stub in
 * INTEGRATION.md).  Each entry point names the reference code it replaces.
 *
 * Conventions: plain pointers and sizes only.  Every pointer is a DEVICE pointer unless its name
 * starts with h_.  The caller owns every buffer; the library allocates nothing and keeps no mutable
 * global state.  All calls are stream-ordered on the cudaStream_t passed as `void* stream`
 * (NULL = default stream), re-entrant across streams.  Return 0 on success, non-zero on error;
 * pmt_last_error() returns a thread-local message.
 *
 * Weights: one flat fp32 buffer holding the MATERIALISED (constraint-applied) parameters in
 * ArtifactModel.named_parameters() order (SURVEY.md Appendix B); PmtModelDesc carries the offsets.
 * Gradients come back in a flat buffer of the same layout.
 */
#ifndef PERMUTECT_B200_H
#define PERMUTECT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMT_ABI_VERSION 4
#define PMT_MAX_MLP_OPS 16
#define PMT_MAX_BLOCKS 12
#define PMT_MAX_CNN_OPS 16
#define PMT_MAX_DIM 64      /* widest per-read activation / layer width */
#define PMT_MAX_INFO_DIM 128 /* widest info-feature input */
#define PMT_MAX_FEAT 32     /* final feature dimension E */
#define PMT_MAX_CLUSTERS 14 /* K; K+2 log-likelihood columns <= 16 */
#define PMT_TILE_ROWS 128   /* reads per CTA tile */

/* PmtLinearOp.flags */
#define PMT_OP_POST_SELU 1   /* SELU applied to the output                      (mlp.py:61-62) */
#define PMT_OP_SKIP_BEGIN 2  /* first layer of a DenseSkipBlock: input is SELU(x) (mlp.py:8-22) */
#define PMT_OP_SKIP_END 4    /* last layer of a DenseSkipBlock: x <- x + alpha * y             */

/* One nn.Linear of an MLP program (reference: permutect/architecture/mlp.py:25-76). */
typedef struct PmtLinearOp {
  int32_t in_dim, out_dim;
  int32_t w_off, b_off;   /* offsets (floats) into the flat weight buffer; weight is [out][in] */
  int32_t alpha_off;      /* DenseSkipBlock.alpha (valid when PMT_OP_SKIP_END) */
  int32_t flags;
} PmtLinearOp;

/* PmtCnnOp.kind */
#define PMT_CNN_CONV 1
#define PMT_CNN_POOL 2
#define PMT_CNN_LINEAR 3   /* after flatten; in_ch = channels*length, out_ch = out_features */
/* PmtCnnOp.act */
#define PMT_ACT_NONE 0
#define PMT_ACT_SELU 1
#define PMT_ACT_LEAKY_RELU 2

/* One layer of DNASequenceConvolution (reference: dna_sequence_convolution.py:57-111).
 * An activation that follows a conv (possibly after max-pools, with which any monotone activation
 * commutes exactly) is folded into that conv's `act`. */
typedef struct PmtCnnOp {
  int32_t kind, in_ch, out_ch, ksize, stride, in_len, out_len, act;
  int32_t w_off, b_off;   /* conv weight [out][in][k]; linear weight [out][in_ch] */
} PmtCnnOp;

/* Parameter offsets of one GatedRefAltMLPBlock (reference: gated_mlp.py:148-251). */
typedef struct PmtBlockOffsets {
  int32_t ln_w, ln_b;               /* norm (shared by ref and alt, quirk Q4) */
  int32_t p1_ref_w, p1_ref_b, p1_alt_w, p1_alt_b;
  int32_t alpha_ref, alpha_alt, beta_ref, beta_alt, gamma;
  int32_t regularizer;              /* sgu.ref_regularizer [d_ffn/2] */
  int32_t ln2_w, ln2_b;             /* sgu.norm */
  int32_t reg_weight;               /* materialised exp(reg_weight.original); kernel adds 0.25 (gated_mlp.py:237) */
  int32_t p2_ref_w, p2_ref_b, p2_alt_w, p2_alt_b;
} PmtBlockOffsets;

typedef struct PmtModelDesc {
  int32_t abi_version;
  int32_t n_read_features;   /* decoded width F = 8*7 + (read_row_bytes - 7) */
  int32_t read_row_bytes;    /* bytes per compressed read (12) */
  int32_t n_info_features, hap_len; /* hap_len = L, each variant has 2L haplotype codes */
  int32_t d_read, d_info, d_seq, d_model, d_ffn, n_blocks, d_feat, n_clusters;
  int32_t n_read_ops, n_info_ops, n_red_ops, n_cnn_ops;
  PmtLinearOp read_ops[PMT_MAX_MLP_OPS];   /* read_embedding   (artifact_model.py:142) */
  PmtLinearOp info_ops[PMT_MAX_MLP_OPS];   /* info_embedding   (artifact_model.py:147) */
  PmtLinearOp red_ops[PMT_MAX_MLP_OPS];    /* reducer          (artifact_model.py:164) */
  PmtCnnOp cnn_ops[PMT_MAX_CNN_OPS];       /* haplotypes_cnn   (artifact_model.py:152) */
  PmtBlockOffsets blocks[PMT_MAX_BLOCKS];  /* ref_alt_reads_encoder (artifact_model.py:161) */
  int32_t translation, rotation;           /* pre_clustering_transform: t[E], Q[E][E] (f = Q (y + t)) */
  int32_t sigma_e, unit_ke, tau_k, logw_k, mu_k, emg_sigma_k, lambda_k; /* feature_clustering, materialised */
  int32_t n_params;                        /* length of the flat buffer */
} PmtModelDesc;

/* PmtBatch.reads_kind / info_kind / hap_kind */
#define PMT_READS_U8 0    /* compressed rows [R][read_row_bytes] (datum.py:27, batch.py:51-56) */
#define PMT_READS_F32 1   /* decoded rows [R][F] float32 */
#define PMT_READS_F16 2   /* decoded rows [R][F] float16 */
#define PMT_F32 0
#define PMT_F16 1
#define PMT_I16 0
#define PMT_I64 1

/* One batch of ragged read sets, laid out as the reference's Batch (batch.py:41-62):
 * all ref reads of all variants, then all alt reads.  Row n of the batch is source row
 * read_indices[n] when read_indices != NULL (DownsampledBatch.get_reads_re, batch.py:458-459;
 * indices are consumed verbatim, quirk Q1), else row n. */
typedef struct PmtBatch {
  int32_t n_variants;
  int32_t reads_kind, info_kind, hap_kind;
  int64_t n_rows;              /* host-side upper bound of total_ref + total_alt (grid sizing hint; <= 0: unknown).
                                  The kernels take the exact totals from ref_off[B] / alt_off[B]. */
  int64_t total_ref;
  int64_t max_rows_per_variant;/* >= max_b(ref_count+alt_count); sizes the long-set workspace */
  const void* reads;
  const int64_t* read_indices; /* NULL or [n_rows] */
  const int64_t* ref_off;      /* [B+1] exclusive prefix sums of ref counts */
  const int64_t* alt_off;      /* [B+1] exclusive prefix sums of alt counts */
  const void* info;            /* [B][info_stride], first n_info_features used */
  int64_t info_stride;
  const void* haplotypes;      /* [B][hap_stride], first 2*hap_len used; codes 0..4 */
  int64_t hap_stride;
} PmtBatch;

/* Replaces BatchOutput (artifact_model.py:38-73) minus the balancer weights. Any pointer may be NULL. */
typedef struct PmtOutputs {
  float* logits_bk;       /* [B][K+2]  feature_clustering.py:82-119 */
  float* logits_b;        /* [B]       20*tanh(raw/20), feature_clustering.py:121-135 */
  float* outlier_logits_b;/* [B]       artifact_model.py:62-73 */
  float* alt_means_be;    /* [B][E]    features_be, artifact_model.py:291 */
  float* ref_means_be;    /* [B][E]    ref_features_be, artifact_model.py:292 */
  float* info_seq_be;     /* [B][d_info+d_seq]  artifact_model.py:244-246 (ref_seq embedding = last d_seq columns) */
  float* final_re;        /* [n_rows][E] per-read final features (calculate_features, artifact_model.py:261-265) */
} PmtOutputs;

/* Upstream gradients for pmt_backward (dL/d of the PmtOutputs fields that carry gradient). NULL = zero. */
typedef struct PmtOutGrads {
  const float* d_logits_bk;   /* [B][K+2] */
  const float* d_alt_means_be;/* [B][E] */
  const float* d_ref_means_be;/* [B][E] */
  const float* info_seq_be;   /* [B][d_info+d_seq] PmtOutputs.info_seq_be saved from the forward of the same batch and
                                 weights, or NULL: the per-variant embeddings are then recomputed */
  const void* saved;          /* the buffer pmt_forward_train filled for the same batch and weights, or NULL: the backward
                                 recomputes the forward (in bounded passes) itself */
} PmtOutGrads;

const char* pmt_last_error(void);
int pmt_abi_version(void);

/* Training without recompute.  pmt_forward_train is pmt_forward that additionally leaves, in `saved`, everything the
 * tensor-core backward would otherwise recompute (the tile list, every layer's operand panels of every tile, the haplotype
 * CNN's activations); pmt_backward takes the same buffer through PmtOutGrads.saved and skips its recompute passes.
 * pmt_train_saved_bytes: bytes of `saved` for this batch, or 0 when the current precision mode / model shape has no such
 * path or the buffer would pass 16 GB (0.7 MB per 128 reads) -- call pmt_forward and leave PmtOutGrads.saved NULL then. */
size_t pmt_train_saved_bytes(const PmtModelDesc* desc, const PmtBatch* batch);
int pmt_forward_train(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                      void* workspace, size_t workspace_bytes, void* saved, size_t saved_bytes, void* stream);

/* Bytes of device workspace pmt_forward / pmt_backward need for this model and batch shape. */
size_t pmt_workspace_size(const PmtModelDesc* desc, const PmtBatch* batch, int for_backward);

/* Forward: ArtifactModel.calculate_features + FeatureClustering.calculate_logits + set means
 * (artifact_model.py:239-297). */
int pmt_forward(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                void* workspace, size_t workspace_bytes, void* stream);

/* Same as pmt_forward, for repeated inference with unchanged weights: skips rebuilding the packed weight images.
 * Contract: the previous call on this workspace was pmt_forward or pmt_forward_prepared with the SAME desc, weights
 * contents, precision mode and workspace base address (the images live at fixed offsets from the base; batches of any
 * size may follow each other), and nothing else wrote to the workspace in between (pmt_backward does). */
int pmt_forward_prepared(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                         void* workspace, size_t workspace_bytes, void* stream);

/* Backward of pmt_forward (autograd of artifact_model.py:239-297): accumulates nothing, WRITES
 * d_weights[n_params] (gradient w.r.t. the materialised flat weights).  Read sets of any length: sets longer than a
 * tile (PMT_TILE_ROWS rows) are walked in chunks, like the forward.  Bitwise reproducible from run to run. */
int pmt_backward(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutGrads* grads,
                 float* d_weights, void* workspace, size_t workspace_bytes, void* stream);

/* Backward of the clustering head alone: the gradient of pmt_forward's outputs w.r.t. the rotation, the translation and
 * the feature-clustering parameters (translation, rotation, sigma_e, unit_ke, tau_k, mu_k, emg_sigma_k, lambda_k, logw_k),
 * for steps in which nothing upstream of the rotation trains (calibration epochs, model_training.py:145-147).  It reads
 * only final_re [n_rows][E], the per-read final features PmtOutputs.final_re of a pmt_forward of the same batch and
 * weights, and grads->d_logits_bk / d_alt_means_be / d_ref_means_be (info_seq_be and saved are not read).  WRITES
 * d_weights[n_params]: the head's slots, exact zeros everywhere else.  Takes every shape pmt_forward takes (none of the
 * trunk backward's limits apply), reads all sizes from the device offsets (no host synchronisation) and is bitwise
 * reproducible from run to run. */
size_t pmt_head_backward_workspace_size(const PmtModelDesc* desc);
int pmt_head_backward(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const float* final_re,
                      const PmtOutGrads* grads, float* d_weights, void* workspace, size_t workspace_bytes, void* stream);

/* Arithmetic mode of the dense layers of the read path (process-wide; default PMT_PRECISION_FP32).
 *   FP32    FP32 FMA pipe (SIMT); forward and backward.
 *   TF32X3  tcgen05 tensor cores, TF32 with a hi/lo split of both operands (3 MMAs, ~2^-21 relative error):
 *           the fp32-parity mode on tensor cores.
 *   TF32    tcgen05 tensor cores, plain TF32 (10-bit mantissa); logits are NOT within 1e-3 of the reference,
 *           tolerance stated separately (DESIGN.md).
 * In both tensor-core modes the backward runs on the tensor cores too, for models inside their envelope
 * (pmt_backward_kernels): it recomputes the forward in split precision and multiplies the gradients in TF32 with fp32
 * accumulation, in either mode.  Models outside it take the FP32 backward. */
#define PMT_PRECISION_FP32 0
#define PMT_PRECISION_TF32X3 1
#define PMT_PRECISION_TF32 2
int pmt_set_precision(int mode);
int pmt_get_precision(void);
/* Which kernels the backward of this model runs in the CURRENT precision mode: *reads_tc = 1 when the read path's backward
 * is the tcgen05 kernel (pmt_tc_bwd.cu), *cnn_tc = 1 when the haplotype CNN's is the tensor-core kernel (pmt_cnn_bwd.cu);
 * 0 = the FP32 SIMT kernel (FP32 mode, or a shape outside the tensor-core kernel's envelope).  Returns non-zero on a bad
 * descriptor. */
int pmt_backward_kernels(const PmtModelDesc* desc, int32_t* reads_tc, int32_t* cnn_tc);

/* Measurement hook (no reference counterpart): when both are non-NULL, the next pmt_forward /
 * pmt_backward calls of this process record these cudaEvent_t around their dominant kernel
 * (reads_forward_kernel / reads_backward_kernel) on the call's stream.  Pass NULLs to disarm. */
int pmt_set_profile_events(void* start_event, void* stop_event);

/* DownsampledBatch.__init__ (batch.py:383-439) on the device, in two stream-ordered steps with an
 * exclusive scan of the new counts (caller-side) in between.  Keep decisions are a counter-based hash of
 * (seed, read row) compared with the per-variant keep fractions; one alt read per variant is always
 * kept (batch.py:418-425, `random_int` plays the role of the reference's randint(0, 100)).
 * read_indices receives the kept ref rows followed by the kept alt rows; alt entries are NOT offset by
 * the ref-block size unless offset_alt_rows != 0 (reference behaviour, quirk Q1, batch.py:436-439). */
int pmt_downsample_counts(const int64_t* ref_off, const int64_t* alt_off, const float* ref_fracs, const float* alt_fracs,
                          int32_t n_variants, uint64_t seed, int32_t random_int, int64_t* new_ref_counts,
                          int64_t* new_alt_counts, void* stream);
int pmt_downsample_fill(const int64_t* ref_off, const int64_t* alt_off, const float* ref_fracs, const float* alt_fracs,
                        int32_t n_variants, uint64_t seed, int32_t random_int, const int64_t* new_ref_off,
                        const int64_t* new_alt_off, int32_t offset_alt_rows, int64_t* read_indices, void* stream);

/* Batch.__init__ decode (batch.py:51-56, plain_text_data.py:510-511): compressed rows -> [R][F] float32. */
int pmt_decode_reads(const uint8_t* reads_u8, int64_t n_rows, int32_t row_bytes, float* out, void* stream);

/* ---- fused loss head -------------------------------------------------------------------------------
 * Replaces ArtifactModel.compute_batch_losses (artifact_model.py:299-325) together with
 * compute_alt_count_losses (:276-279), compute_source_prediction_losses (:267-274), the gradient reversal of the
 * two adversarial heads (gradient_reversal/functional.py:6-22) and the autograd backward of all of it. */
#define PMT_MAX_HEAD_DIM 32   /* widest layer / input of an adversarial head; also the largest number of sources */

typedef struct PmtLossDesc {
  int32_t d_feat;                          /* E: width of features_be */
  int32_t n_sources;                       /* outputs of the source head */
  int32_t n_alt_ops, n_src_ops;            /* n_src_ops == 0: the source loss is identically zero (num_sources == 1) */
  PmtLinearOp alt_ops[PMT_MAX_MLP_OPS];    /* alt_count_predictor.wrapped_module, offsets into the flat weight buffer */
  PmtLinearOp src_ops[PMT_MAX_MLP_OPS];    /* source_predictor.wrapped_module */
  float alt_reversal, src_reversal;        /* GradientReversal.alpha of each head */
  float max_outlier_logit;                 /* MAX_LOGIT clip of the unsupervised loss (artifact_model.py:32,314) */
  float max_alt_count;                     /* alt-count regression target = alt_count / max_alt_count (:278) */
  int32_t n_params;                        /* length of the flat weight / gradient buffers */
} PmtLossDesc;

typedef struct PmtLossBatch {
  int32_t n_variants;
  int32_t label_col, source_col, alt_count_col; /* columns of the per-variant int16 array (datum.py:51-60) */
  const int16_t* int_array;                /* [B][int_stride] */
  int64_t int_stride;
  const int64_t* alt_counts;               /* [B] alt counts when they differ from the int array (DownsampledBatch), else NULL */
  const float* logits_b;                   /* [B]    BatchOutput.logits_b */
  const float* outlier_logits_b;           /* [B]    BatchOutput.outlier_binary_logits */
  const float* features_be;                /* [B][E] BatchOutput.features_be */
  const float* weights_b;                  /* [B] or NULL (= 1) BatchOutput.weights */
  const float* source_weights_b;           /* [B] or NULL (= 1) BatchOutput.source_weights */
} PmtLossBatch;

/* BatchLosses fields (artifact_model.py:76-90); any pointer may be NULL. */
typedef struct PmtLossOutputs {
  float* supervised_b; float* unsupervised_b; float* alt_count_b; float* source_b; float* total_b;
} PmtLossOutputs;

/* Upstream gradients of the five per-variant loss vectors; NULL = zero. */
typedef struct PmtLossGrads {
  const float* g_supervised_b; const float* g_unsupervised_b; const float* g_alt_count_b; const float* g_source_b;
  const float* g_total_b;
} PmtLossGrads;

int pmt_losses_forward(const PmtLossDesc* desc, const float* weights, const PmtLossBatch* batch, const PmtLossOutputs* out,
                       void* stream);
size_t pmt_losses_workspace_size(const PmtLossDesc* desc, int32_t n_variants);
/* WRITES d_logits_b[B], d_outlier_logits_b[B], d_features_be[B][E] (any may be NULL) and d_weights[n_params]
 * (zero outside the two heads' parameters).  Deterministic: bitwise identical from run to run. */
int pmt_losses_backward(const PmtLossDesc* desc, const float* weights, const PmtLossBatch* batch, const PmtLossGrads* grads,
                        float* d_logits_b, float* d_outlier_logits_b, float* d_features_be, float* d_weights,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- flat optimiser step ---------------------------------------------------------------------------
 * Replaces misc_utils.backpropagate's clip_grad_norm_(max_norm=1.0) + AdamW.step (misc_utils.py:125-129;
 * optimiser built at model_training.py:68-72) for a model whose parameters are views of one flat fp32 buffer.
 * grads is the flat gradient in the same layout (already summed across ranks for data-parallel training);
 * mask (NULL = all ones) marks entries whose parameter has a gradient -- masked-out entries are not touched, as
 * torch skips parameters whose .grad is None.  step_count[n] counts the updates each entry has taken (torch keeps one
 * step counter per parameter; bias corrections use it).  max_norm <= 0 disables clipping.  The total gradient
 * norm (before clipping) is written to total_norm_out when non-NULL.  Two launches, no host synchronisation. */
size_t pmt_adamw_workspace_size(void);
int pmt_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int32_t* step_count,
                   const float* mask, int64_t n, float lr, float beta1, float beta2, float eps, float weight_decay, float max_norm,
                   float* total_norm_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- rotation matrix of the orthogonal parametrisation --------------------------------------------------
 * EuclideanTransformation's rotation (architecture/euclidean_transformation.py:11-14) is a torch orthogonal
 * parametrisation with the matrix-exponential map: Q = base @ exp(tril(X) - tril(X)^T).  x, base (may be NULL), q, d_q,
 * d_x: [n][n] fp32 on the device, n <= 16.  Forward and its vector-Jacobian product, each one single-CTA launch
 * (the torch formulation costs ~135 tensor ops of host time per training step). */
int pmt_orthogonal_forward(const float* x, const float* base, int32_t n, float* q, void* stream);
int pmt_orthogonal_backward(const float* x, const float* base, const float* d_q, int32_t n, float* d_x, void* stream);

/* ---- constraint maps of the parametrised tensors -------------------------------------------------------
 * The reference registers torch parametrisations on a dozen tensors (utils/parameterizations.py: PositiveNumber = exp,
 * BoundedNumber = size * sigmoid + min, UnitVector = x / |x| per row, LogWeights = log_softmax); the kernels read the
 * CONSTRAINED values from the flat buffer.  Forward: w = raw with every group replaced by its constrained value; backward:
 * g = d_w with every group replaced by its vector-Jacobian product.  mask[n] marks the entries that belong to a group
 * (the others are copied); groups live in device memory.  One launch each, no host synchronisation.  The rotation of
 * the orthogonal parametrisation is separate (pmt_orthogonal_forward / _backward): mark its entries in the mask and
 * fill them afterwards. */
#define PMT_CONSTRAINT_EXP 0
#define PMT_CONSTRAINT_BOUNDED 1
#define PMT_CONSTRAINT_UNIT 2
#define PMT_CONSTRAINT_UNIT_TWICE 3   /* feature_clustering.py:24 normalises the unit directions once more */
#define PMT_CONSTRAINT_LOGSOFTMAX 4
typedef struct PmtConstraintGroup {
  int32_t type, off, rows, cols;
  float a, b;                         /* BoundedNumber: size, minimum */
} PmtConstraintGroup;
int pmt_constraints_forward(const float* raw, const uint8_t* mask, int64_t n, const PmtConstraintGroup* groups, int32_t n_groups,
                            float* w, void* stream);
int pmt_constraints_backward(const float* raw, const float* w, const float* d_w, const uint8_t* mask, int64_t n,
                             const PmtConstraintGroup* groups, int32_t n_groups, float* g, void* stream);

/* ---- inference caller tail --------------------------------------------------------------------------
 * Replaces the per-variant Python loop of generate_posterior_data (tools/filter_variants.py:302-320): for every
 * variant, int_out[n_int_columns] = its int16 record with REF_COUNT / ALT_COUNT zeroed, float_out[6 + d_feat] (fp32,
 * the dtype np.hstack gives the Datum, datum.py:239-240, and the posterior memory map is created with,
 * memory_mapped_data.py:321) = the six fp16 scalars, slot 5 (CACHED_ARTIFACT_LOGIT) = the fp16-rounded artifact
 * logit (datum.py:207-208, quirk Q6), then the embedding row of features_be. */
int pmt_pack_posterior(const int16_t* int_array, int64_t int_stride, int32_t n_int_columns, const void* float_array_f16,
                       int64_t float_stride, const float* logits_b, const float* features_be, int32_t d_feat,
                       int32_t n_variants, int16_t* int_out, float* float_out, void* stream);

/* ---- posterior model (inference half) ------------------------------------------------------------------
 * Replaces PosteriorModel.log_posterior_and_ingredients (architecture/posterior_model.py:69-99) with
 * PosteriorModelPriors.log_priors_bc (posterior_model_priors.py:121-139) and
 * PosteriorModelSpectra.spectra_log_likelihoods_bc (spectra/posterior_model_spectra.py:78-124) for a batch of posterior
 * records: int_array[n][int_stride] int16 (VARIANT_TYPE 3, ORIGINAL_DEPTH 5, ORIGINAL_ALT_COUNT 6,
 * ORIGINAL_NORMAL_DEPTH 7, ORIGINAL_NORMAL_ALT_COUNT 8, haplotype codes from hap_start), float_array[n][float_stride]
 * (SEQ_ERROR_LOG_LK 0, NORMAL_SEQ_ERROR_LOG_LK 1, ALLELE_FREQUENCY 2, MAF 3, NORMAL_MAF 4, CACHED_ARTIFACT_LOGIT 5;
 * datum.py:51-81).  `params`: pmt_posterior_param_count(K) floats of CONSTRAINED values in this order: cell
 * fractions cf_k[K], log weights[K], log background weight, log non-background weight, background alpha, beta,
 * artifact alpha_dv[3][5], beta_dv[3][5], normal-artifact alpha_dv[3][5], beta_dv[3][5], mean_multiplier_v[5],
 * concentration_v[5], log_priors_vc[5][5], somatic_snv_log_priors_rrra[5][5][5][5].  Outputs are [n][5] in Call order
 * (SOMATIC, ARTIFACT, SEQ_ERROR, GERMLINE, NORMAL_ARTIFACT); any may be NULL. */
#define PMT_POSTERIOR_MAX_COMPONENTS 16
typedef struct PmtPosteriorDesc {
  int32_t n_components;                     /* K of SomaticSpectrum (somatic_spectrum.py:46) */
  int32_t hap_start, hap_len;               /* column of the first haplotype code, bases per haplotype (ref then alt) */
  int32_t no_germline_mode;                 /* posterior_model.py:37 */
  int32_t use_context_dependent_snv_priors; /* posterior_model_priors.py:99-103 */
  float het_beta;                           /* < 0: None (binomial het likelihood, posterior_model_spectra.py:46-51) */
} PmtPosteriorDesc;
typedef struct PmtPosteriorOutputs {
  float* log_priors_bc;
  float* spectra_log_lks_bc;
  float* normal_log_lks_bc;
  float* log_posteriors_bc;
  float* posterior_probabilities_bc;        /* softmax of log_posteriors_bc (posterior_model.py:51-56) */
} PmtPosteriorOutputs;
int pmt_posterior_param_count(int32_t n_components);
int pmt_posterior_log_posteriors(const PmtPosteriorDesc* desc, const float* params, const int16_t* int_array,
                                 int64_t int_stride, const void* float_array, int32_t float_kind, int64_t float_stride,
                                 int32_t n_variants, const PmtPosteriorOutputs* out, void* stream);

/* One E step of PosteriorModel.learn_priors_and_spectra (posterior_model.py:131-151) over a batch: loss_out[1] =
 * -mean_b logsumexp_c log_posteriors_bc; grads_out[2K + 70] = its gradient w.r.t. the CONSTRAINED spectra tensors in
 * the order cf_k[K], log_weights_k[K], artifact alpha_dv[3][5], beta_dv[3][5], normal-artifact alpha_dv[3][5],
 * beta_dv[3][5], mean_multiplier_v[5], concentration_v[5] (the caller chains the parametrisations);
 * posterior_totals_tc[5][5] += sum of the posteriors by variant type (:143), somatic_snv_totals_rrra /
 * snv_context_totals_rrra [5][5][5][5] += the SNV context totals (posterior_model_priors.py:105-119).  Any output may be
 * NULL.  Loss, gradients and posterior_totals_tc are summed in a fixed order (bitwise reproducible); the context totals
 * use atomics. */
size_t pmt_posterior_fit_workspace_size(int32_t n_variants, int32_t n_components);
int pmt_posterior_fit_step(const PmtPosteriorDesc* desc, const float* params, const int16_t* int_array,
                           int64_t int_stride, const void* float_array, int32_t float_kind, int64_t float_stride,
                           int32_t n_variants, float* loss_out, float* grads_out, float* posterior_totals_tc,
                           float* somatic_snv_totals_rrra, float* snv_context_totals_rrra, void* workspace,
                           size_t workspace_bytes, void* stream);

/* One pass of PosteriorModel.learn_priors_and_spectra's batch loop (posterior_model.py:128-151) in one launch: the
 * records [n_records] are taken in order in batches of batch_size (the last may be shorter), and every batch gets the E
 * step of pmt_posterior_fit_step and then one step of torch.optim.Adam (betas 0.9 / 0.999, eps 1e-8, no weight decay,
 * bias corrections from the step count) on the RAW spectra entries, the constrained values of the next batch being
 * re-materialised through the parametrisations (cf_k, mean_multiplier_v: BoundedNumber(0, 1); log_weights_k: LogWeights;
 * artifact and normal-artifact alpha_dv / beta_dv, concentration_v: PositiveNumber).  `params`: as for
 * pmt_posterior_log_posteriors, the constrained values of raw_params at the start of the pass; its priors and background
 * entries stay fixed for the pass.  raw_params, adam_m, adam_v [2K + 70] (in / out) in the order of
 * pmt_posterior_fit_step's grads_out; adam_step[1] (in / out) += the number of batches.  batch_losses_out[number of
 * batches] = every batch's loss.  posterior_totals_tc, somatic_snv_totals_rrra, snv_context_totals_rrra += the pass's
 * E-step totals, as pmt_posterior_fit_step adds them (any may be NULL).  Every sum has a fixed order and no atomics:
 * the pass is bitwise reproducible.  A cluster of up to 16 CTAs, so up to 16 SMs, walks the batches, its CTAs sharing
 * each batch's records through distributed shared memory; every width gives the same bits (pmt_posterior_fit_ctas
 * reports the width).  workspace: pmt_posterior_fit_pass_workspace_size(K) bytes (0 for a K outside
 * 1..PMT_POSTERIOR_MAX_COMPONENTS). */
size_t pmt_posterior_fit_pass_workspace_size(int32_t n_components);
int pmt_posterior_fit_pass(const PmtPosteriorDesc* desc, const float* params, float* raw_params, float* adam_m, float* adam_v,
                           int64_t* adam_step, double learning_rate, const int16_t* int_array, int64_t int_stride,
                           const void* float_array, int32_t float_kind, int64_t float_stride, int64_t n_records,
                           int32_t batch_size, float* batch_losses_out, float* posterior_totals_tc,
                           float* somatic_snv_totals_rrra, float* snv_context_totals_rrra, void* workspace,
                           size_t workspace_bytes, void* stream);

/* The passes of many independent fits (a cohort's samples, each with its own model and records) in one launch: one
 * cluster of CTAs per problem (up to 16 SMs each), each running exactly pmt_posterior_fit_pass's pass on its own
 * arguments, so problem i ends with the bits pmt_posterior_fit_pass gives for it alone.  A sample's fit is a sequential
 * chain of Adam steps; the clusters are as wide as lets every problem's cluster be resident at once (one CTA each from
 * as many problems as SMs on, more problems than SMs run in waves).  Problems may differ in
 * every field: K, het_beta, no-germline mode, context priors, record count, batch size, fp16 / fp32 floats and strides,
 * learning rate, which totals are NULL.  Every argument check of pmt_posterior_fit_pass applies to every problem, all
 * before anything is enqueued; a refusal names the problem's index.  `h_problems` is a HOST array of n_problems >= 1;
 * the call copies it into the workspace (stream-ordered, the host array may be reused once the call returns).
 * workspace: pmt_posterior_fit_pass_many_workspace_size(n_problems, largest K of the problems) bytes (0 for
 * n_problems < 1 or a K outside 1..PMT_POSTERIOR_MAX_COMPONENTS): the problem table and each problem's context scratch. */
typedef struct PmtPosteriorFitProblem {
  PmtPosteriorDesc desc;
  const float* params;
  float* raw_params;
  float* adam_m;
  float* adam_v;
  int64_t* adam_step;
  double learning_rate;
  const int16_t* int_array;
  int64_t int_stride;
  const void* float_array;
  int32_t float_kind;
  int64_t float_stride;
  int64_t n_records;
  int32_t batch_size;
  float* batch_losses_out;
  float* posterior_totals_tc;               /* these three may be NULL, as for pmt_posterior_fit_pass */
  float* somatic_snv_totals_rrra;
  float* snv_context_totals_rrra;
} PmtPosteriorFitProblem;
size_t pmt_posterior_fit_pass_many_workspace_size(int32_t n_problems, int32_t max_components);
int pmt_posterior_fit_pass_many(const PmtPosteriorFitProblem* h_problems, int32_t n_problems, void* workspace, size_t workspace_bytes,
                                void* stream);
/* The cluster width (CTAs per problem: 1, 2, 4, 8 or 16) with which pmt_posterior_fit_pass_many runs these n_problems
 * problems, or pmt_posterior_fit_pass a single one: the largest width that gives every CTA at least 16 records of the
 * largest batch (a warp each) and lets every problem's cluster be resident at once, and 1 from as many problems as SMs
 * on.  The width never changes a result.  The environment variable PMT_POSTERIOR_CTAS=n (tests and measurements) forces
 * the width n of both passes; any other value than the five widths makes them, and this query, refuse.  Returns 0 with
 * pmt_last_error() on a refusal: the fit-pass checks of every problem apply (the problem's index is named), and the
 * query needs the device the passes would run on. */
int pmt_posterior_fit_ctas(const PmtPosteriorFitProblem* h_problems, int32_t n_problems);

/* The context-dependent SNV-prior fit of the posterior model's M step (architecture/snv_context_priors.py,
 * fit_mutation_rates_sc) for n independent problems in one launch, one CTA each, float64 throughout: the mean-field fit
 * of the hierarchical substitution x context model to problem i's rounded totals by the algorithm of torch.optim.LBFGS
 * (strong-Wolfe line search, max_iter 300) over the sample-average ELBO of the 64 draws `elbo_draws`, then
 * rates_out[i][12][16] = E_q[rate_sc], the mean over the 1000 draws `mean_draws`.  total_sc, snv_sc: contiguous
 * [n][12][16] (snv is clamped to total, as the host fit does); elbo_draws [64][194] and mean_draws [1000][194]: the
 * standard-normal tables of the host fit (_sobol_normal(64, 194, 1234) and _sobol_normal(1000, 194, 4321)).  Optional
 * outputs (may be NULL): mu_out, log_sigma_out [n][194], the fitted variational parameters; n_iter_out,
 * func_evals_out [n], the optimiser's iteration and objective-evaluation counts.  Every reduction has a fixed order and
 * problems do not interact: problem i gives the same bits whatever else is in the launch.  workspace:
 * pmt_snv_context_fit_workspace_size(n) bytes (0 for n < 1), the problems' L-BFGS histories.  Refused before anything
 * is enqueued: n < 1, a NULL required pointer, a short workspace. */
size_t pmt_snv_context_fit_workspace_size(int32_t n);
int pmt_snv_context_fit_many(int32_t n, const double* total_sc, const double* snv_sc, const double* elbo_draws,
                             const double* mean_draws, double* rates_out, double* mu_out, double* log_sigma_out,
                             int32_t* n_iter_out, int32_t* func_evals_out, void* workspace, size_t workspace_bytes,
                             void* stream);

/* ---- batch assembly from the dataset memory maps ----------------------------------------------------
 * Replaces the row re-stacking of Batch.__init__ (batch.py:41-62) for batches cut from a MemoryMappedData
 * (memory_mapped_data.py:36-58, reads_dataset.py:109-196): the reads memory map holds, variant after variant, the ref
 * rows then the alt rows; a batch is shipped as the contiguous slice of that map and read_indices[n_rows] receives,
 * for every batch row (all ref rows by variant, then all alt rows, batch.py:45-47), its row in the slice.
 * ref_off / alt_off: exclusive prefix sums [n_variants + 1] of the variants' counts (device). */
int pmt_dataset_read_indices(const int64_t* ref_off, const int64_t* alt_off, int32_t n_variants, int64_t* read_indices,
                             void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PERMUTECT_B200_H */
