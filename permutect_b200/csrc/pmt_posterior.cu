// PosteriorModel.log_posterior_and_ingredients as one kernel (SURVEY §8 f3; reference posterior_model.py:69-99).
//
// One thread per variant: log priors (posterior_model_priors.py:121-139), the five spectra log-likelihoods
// (posterior_model_spectra.py:78-124: somatic_spectrum.py:74-98, artifact_spectra.py:45-55,
// normal_artifact_spectrum.py:38-58, germline :18-58), the matched-normal table, and their sum with the cached artifact
// logit.  The reference builds ~25 [B] or [B, K, 100] temporaries per call; here a variant's 5 x 100 binomial terms of
// the somatic mixture live in registers and nothing but the requested [B, 5] tables touches HBM.
// fit_pass_kernel runs a whole pass of the fit's batch loop (E step, parametrisation VJP, Adam) on one cluster of up to 16
// CTAs on the same per-record device functions; fit_pass_many_kernel runs the passes of independent problems (one per
// sample) a cluster each.
#include <cooperative_groups.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>

#include <algorithm>
#include <cstdio>
#include <vector>

#include "../../include/permutect_b200.h"
#include "pmt_host.h"

namespace post {

constexpr int N_CALLS = 5, SOMATIC = 0, ARTIFACT = 1, SEQ_ERROR = 2, GERMLINE = 3, NORMAL_ARTIFACT = 4;   // utils/enums.py Call
constexpr int N_TYPES = 5, N_DEPTH_BINS = 3;
constexpr int N_INTERP = 100;   // torch.arange(0.001, 0.999, 0.01), stats_utils.py:183

struct Online {   // streaming logsumexp
  float m = -INFINITY, s = 0.f;
  __device__ __forceinline__ void add(float v) {
    if (v > m) { s = s * expf(m - v) + 1.f; m = v; }
    else s += expf(v - m);
  }
  __device__ __forceinline__ float value() const { return m + logf(s); }
};

struct OnlineD {   // streaming logsumexp that also carries sum_j softmax_j * q_j (q_j: a derivative attached to term j)
  float m = -INFINITY, s = 0.f, d = 0.f;
  __device__ __forceinline__ void add(float v, float q) {
    if (v > m) { const float sc = expf(m - v); s = s * sc + 1.f; d = d * sc + q; m = v; }
    else { const float e = expf(v - m); s += e; d += e * q; }
  }
  __device__ __forceinline__ float value() const { return m + logf(s); }
  __device__ __forceinline__ float mean_q() const { return d / s; }
};

// digamma for x > 0: recurrence up to x >= 6, then the asymptotic series
__device__ __forceinline__ float digammaf(float x) {
  float r = 0.f;
  while (x < 6.f) { r -= 1.f / x; x += 1.f; }
  const float i = 1.f / x, i2 = i * i;
  return r + logf(x) - 0.5f * i - i2 * (1.f / 12.f - i2 * (1.f / 120.f - i2 * (1.f / 252.f)));
}
// d beta_binomial / d alpha, d beta (stats_utils.py:29-41)
__device__ __forceinline__ void beta_binomial_grads(float n, float k, float a, float b, float& ga, float& gb) {
  const float common = digammaf(a + b) - digammaf(n + a + b);
  ga = digammaf(k + a) + common - digammaf(a);
  gb = digammaf(n - k + b) + common - digammaf(b);
}

__device__ __forceinline__ float comb_term(float n, float k) { return lgammaf(n + 1.f) - lgammaf(n - k + 1.f) - lgammaf(k + 1.f); }
// stats_utils.py:29-41
__device__ __forceinline__ float beta_binomial(float n, float k, float comb, float a, float b) {
  return comb + lgammaf(k + a) + lgammaf(n - k + b) + lgammaf(a + b) - lgammaf(n + a + b) - lgammaf(a) - lgammaf(b);
}
__device__ __forceinline__ int depth_bin(float d) { return (d >= 10.f ? 1 : 0) + (d >= 20.f ? 1 : 0); }   // artifact_spectra.py:17-24

// posterior_model_spectra.py:18-58
__device__ __forceinline__ float germline(float af, float maf, float alt, float depth, float comb, float het_beta) {
  const float het = 2.f * af * (1.f - af), hom = af * af;
  const float het_prop = het / (het + hom), hom_prop = 1.f - het_prop;
  const float ref = depth - alt;
  float minor, major;
  if (het_beta < 0.f) {
    const float lm = logf(maf), l1m = logf(1.f - maf);
    minor = comb + alt * lm + ref * l1m;
    major = comb + ref * lm + alt * l1m;
  } else {
    minor = major = beta_binomial(depth, alt, comb, het_beta, het_beta);
  }
  const float half = logf(het_prop / 2.f);
  const float hom_ll = logf(hom_prop) + beta_binomial(depth, alt, comb, 98.f, 2.f);
  const float a = half + minor, b = half + major, c = hom_ll;
  const float m = fmaxf(a, fmaxf(b, c));
  return m + logf(expf(a - m) + expf(b - m) + expf(c - m));
}

__device__ __forceinline__ float load_float(const void* p, int kind, long long i) {
  return kind == PMT_F16 ? __half2float(reinterpret_cast<const __half*>(p)[i]) : reinterpret_cast<const float*>(p)[i];
}

constexpr int THREADS = 128, WARPS = THREADS / 32;
constexpr int MAXK = PMT_POSTERIOR_MAX_COMPONENTS;
// slots of the fitting pass, per CTA then summed over CTAs in order: loss, d cf_k, d log_weights_k, d artifact alpha / beta
// [3][5], d normal-artifact alpha / beta [3][5], d mean_multiplier_v, d concentration_v, E-step totals [type][call]
__host__ __device__ constexpr int slot_count(int K) { return 1 + 2 * K + 4 * N_DEPTH_BINS * N_TYPES + 2 * N_TYPES + N_TYPES * N_CALLS; }

struct FitArgs {
  float* partials;                 // [n_blocks][slot_count]
  float* somatic_snv_totals_rrra;  // [5][5][5][5] += posterior(SOMATIC) of SNVs (posterior_model_priors.py:111-119), may be null
  float* snv_context_totals_rrra;  // [5][5][5][5] += 1 per SNV, may be null
};

// Deterministic CTA sum of one slot: warp shuffle tree, lane 0 of each warp owns wsum[warp][slot]
__device__ __forceinline__ void slot_add(float* wsum, int n_slots, int slot, float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) wsum[(threadIdx.x >> 5) * n_slots + slot] += v;
}

// The small constrained parameters (everything but the rrra priors) as the kernels keep them in shared memory, in the
// order of pmt_posterior_log_posteriors' `params`
__host__ __device__ constexpr int small_count(int K) { return 2 * K + 4 + 4 * N_DEPTH_BINS * N_TYPES + 2 * N_TYPES + N_TYPES * N_CALLS; }
struct Spectra {
  const float *cf_k, *logw_k;
  float log_bg, log_non_bg, bg_alpha, bg_beta;
  const float *art_alpha, *art_beta, *na_alpha, *na_beta, *na_mult, *na_conc, *log_priors_vc;
};
__device__ __forceinline__ Spectra spectra_view(const float* sp, int K) {
  Spectra S;
  S.cf_k = sp;
  S.logw_k = S.cf_k + K;
  S.log_bg = S.logw_k[K]; S.log_non_bg = S.logw_k[K + 1]; S.bg_alpha = S.logw_k[K + 2]; S.bg_beta = S.logw_k[K + 3];
  S.art_alpha = S.logw_k + K + 4;
  S.art_beta = S.art_alpha + N_DEPTH_BINS * N_TYPES;
  S.na_alpha = S.art_beta + N_DEPTH_BINS * N_TYPES;
  S.na_beta = S.na_alpha + N_DEPTH_BINS * N_TYPES;
  S.na_mult = S.na_beta + N_DEPTH_BINS * N_TYPES;
  S.na_conc = S.na_mult + N_TYPES;
  S.log_priors_vc = S.na_conc + N_TYPES;
  return S;
}

struct Record {   // the fields of one posterior record the model reads
  const int16_t* ir;
  int vt;
  float depth, alt, ndepth, nalt, seq_err, nseq_err, af, maf, nmaf, logit;
};
__device__ __forceinline__ Record load_record(const int16_t* __restrict__ ints, long long int_stride, const void* __restrict__ floats,
                                              int float_kind, long long float_stride, long long v) {
  Record R;
  R.ir = ints + v * int_stride;
  const long long fo = v * float_stride;
  int vt = R.ir[3];
  R.vt = vt < 0 ? 0 : (vt >= N_TYPES ? N_TYPES - 1 : vt);
  R.depth = (float)R.ir[5]; R.alt = (float)R.ir[6]; R.ndepth = (float)R.ir[7]; R.nalt = (float)R.ir[8];
  R.seq_err = load_float(floats, float_kind, fo + 0); R.nseq_err = load_float(floats, float_kind, fo + 1);
  R.af = load_float(floats, float_kind, fo + 2); R.maf = load_float(floats, float_kind, fo + 3);
  R.nmaf = load_float(floats, float_kind, fo + 4); R.logit = load_float(floats, float_kind, fo + 5);
  return R;
}

// ((ref[c-1] * 5 + ref[c]) * 5 + ref[c+1]) * 5 + alt[c] of an SNV's haplotypes: its cell of the [5][5][5][5] tables
__device__ __forceinline__ int snv_context_cell(const PmtPosteriorDesc& D, const int16_t* ir) {
  const int L = D.hap_len, c = (L - 1) / 2;
  const int16_t* hap = ir + D.hap_start;
  const int i0 = min(max((int)hap[c - 1], 0), 4), i1 = min(max((int)hap[c], 0), 4), i2 = min(max((int)hap[c + 1], 0), 4),
            i3 = min(max((int)hap[c + L], 0), 4);
  return ((i0 * 5 + i1) * 5 + i2) * 5 + i3;
}

// What the E-step gradient of a record needs besides its posteriors
struct Ingredients {
  float non_bg_share;   // share of the non-background mixture in the somatic spectrum
  int db, ndb;          // tumor / normal depth bins
  float a_b, b_b, conc, naf;
};

// Mixture component k's streaming logsumexp over its interpolation points j = j0, j0 + dj, ... < N_INTERP; FIT also
// carries d/d cf_k of every term.  The mixture callers hand the states of all j to `merge` (identity when j0 = 0, dj = 1).
template <bool FIT>
__device__ __forceinline__ OnlineD component_terms(float mafc, float cf, float comb, float alt, float depth, int j0, int dj) {
  const float x1 = mafc * cf, x2 = (1.f - mafc) * cf;
  OnlineD u;
  for (int j = j0; j < N_INTERP; j += dj) {
    const float t = 0.001f + 0.01f * (float)j;
    const float p = x2 * t + x1 * (1.f - t);
    // d/d cf_k of this term: (alt / p - (depth - alt) / (1 - p)) * p / cf_k
    u.add(comb + alt * logf(p) + (depth - alt) * logf(1.f - p), FIT ? (alt - (depth - alt) * p / (1.f - p)) / cf : 0.f);
  }
  return u;
}

struct NoMerge {
  __device__ __forceinline__ OnlineD operator()(const OnlineD& u) const { return u; }
};

// Log priors, the five spectra, the matched-normal table and the log posteriors of one record (posterior_model.py:69-99).
// FIT: mix_term[K] receives the responsibilities of the mixture components, mix_dcf[K] their mean d/d cf_k (Mix: float*,
// or LaneMix in shared memory).
template <bool FIT, class Merge, class Mix>
__device__ __forceinline__ void record_tables(const PmtPosteriorDesc& D, const Spectra& S, const float* snv_rrra, const Record& R,
                                              int j0, int dj, Merge merge, Mix mix_term, Mix mix_dcf, float pri[N_CALLS],
                                              float spec[N_CALLS], float norm[N_CALLS], float post[N_CALLS], Ingredients& I) {
  const int K = D.n_components, vt = R.vt;
  const float depth = R.depth, alt = R.alt, ndepth = R.ndepth, nalt = R.nalt;
  // ---- priors ----
#pragma unroll
  for (int c = 0; c < N_CALLS; ++c) pri[c] = S.log_priors_vc[vt * N_CALLS + c];
  pri[SEQ_ERROR] = 0.f;
  pri[GERMLINE] = D.no_germline_mode ? -9999.f : logf(1.f - (1.f - R.af) * (1.f - R.af));
  if (D.use_context_dependent_snv_priors && vt == 0) pri[SOMATIC] = __ldg(snv_rrra + snv_context_cell(D, R.ir));
  {
    float m = pri[0];
#pragma unroll
    for (int c = 1; c < N_CALLS; ++c) m = fmaxf(m, pri[c]);
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < N_CALLS; ++c) s += expf(pri[c] - m);
    const float lse = m + logf(s);
#pragma unroll
    for (int c = 0; c < N_CALLS; ++c) pri[c] -= lse;
  }

  // ---- spectra ----
  I.non_bg_share = 0.f;
  const float comb = comb_term(depth, alt), ncomb = comb_term(ndepth, nalt);
  {
    const float mafc = fminf(R.maf, 0.49f);                      // somatic_spectrum.py:78
    Online mix;
    for (int k = 0; k < K; ++k) {
      const OnlineD u = merge(component_terms<FIT>(mafc, S.cf_k[k], comb, alt, depth, j0, dj));
      const float term = S.logw_k[k] + u.value() - logf((float)N_INTERP);
      mix.add(term);
      if (FIT) { mix_term[k] = term; mix_dcf[k] = u.mean_q(); }
    }
    const float mixv = mix.value();
    const float a = S.log_non_bg + mixv, b = S.log_bg + beta_binomial(depth, alt, comb, S.bg_alpha, S.bg_beta);
    const float m = fmaxf(a, b);
    spec[SOMATIC] = m + logf(expf(a - m) + expf(b - m));
    if (FIT) {
      I.non_bg_share = expf(a - spec[SOMATIC]);
      for (int k = 0; k < K; ++k) mix_term[k] = expf(mix_term[k] - mixv);     // responsibilities of the components
    }
  }
  const int db = depth_bin(depth), ndb = depth_bin(ndepth);
  spec[ARTIFACT] = beta_binomial(depth, alt, comb, S.art_alpha[db * N_TYPES + vt], S.art_beta[db * N_TYPES + vt]);
  const float na_normal = beta_binomial(ndepth, nalt, ncomb, S.na_alpha[ndb * N_TYPES + vt], S.na_beta[ndb * N_TYPES + vt]);
  const float conc = S.na_conc[vt], naf = nalt / (ndepth + 0.001f);
  const float a_b = 0.001f + naf * S.na_mult[vt] * conc;
  const float b_b = fmaxf(conc - a_b, 0.001f);
  spec[NORMAL_ARTIFACT] = beta_binomial(depth, alt, comb, a_b, b_b);
  spec[SEQ_ERROR] = R.seq_err;
  spec[GERMLINE] = germline(R.af, R.maf, alt, depth, comb, D.het_beta);

  norm[SOMATIC] = R.nseq_err; norm[ARTIFACT] = R.nseq_err; norm[SEQ_ERROR] = R.nseq_err;
  norm[NORMAL_ARTIFACT] = nalt < 1.f ? -9999.f : na_normal;
  norm[GERMLINE] = germline(R.af, R.nmaf, nalt, ndepth, ncomb, D.het_beta);

#pragma unroll
  for (int c = 0; c < N_CALLS; ++c) post[c] = pri[c] + spec[c] + norm[c];
  post[ARTIFACT] += R.logit;
  post[NORMAL_ARTIFACT] += R.logit;
  if (R.logit < 0.f) post[ARTIFACT] = -9999.f;                   // posterior_model.py:90-93
  I.db = db; I.ndb = ndb; I.a_b = a_b; I.b_b = b_b; I.conc = conc; I.naf = naf;
}

// The record's terms of the E step and of the gradient of -sum log evidence (posterior_model.py:139-151), weighted by w,
// handed to sink(slot, value) in slot order (slot_count(K) slots); r[] receives the record's posteriors times w.
template <class Mix, class Sink>
__device__ __forceinline__ void evidence_terms(const Spectra& S, int K, const Record& R, const Ingredients& I, Mix mix_term, Mix mix_dcf,
                                               const float post[N_CALLS], float w, float r[N_CALLS], Sink sink) {
  const int vt = R.vt;
  float pm = post[0];
#pragma unroll
  for (int c = 1; c < N_CALLS; ++c) pm = fmaxf(pm, post[c]);
  float rs = 0.f;
#pragma unroll
  for (int c = 0; c < N_CALLS; ++c) { r[c] = expf(post[c] - pm); rs += r[c]; }
#pragma unroll
  for (int c = 0; c < N_CALLS; ++c) r[c] = w * r[c] / rs;
  int slot = 0;
  sink(slot++, w * (pm + logf(rs)));                                                       // log evidence
  const float ws = r[SOMATIC] * I.non_bg_share;
  for (int k = 0; k < K; ++k) sink(slot + k, ws * mix_term[k] * mix_dcf[k]);
  slot += K;
  for (int k = 0; k < K; ++k) sink(slot + k, ws * mix_term[k]);
  slot += K;
  float ga, gb;
  const int cell = I.db * N_TYPES + vt, ncell = I.ndb * N_TYPES + vt;
  beta_binomial_grads(R.depth, R.alt, S.art_alpha[cell], S.art_beta[cell], ga, gb);
  const float wa = R.logit < 0.f ? 0.f : r[ARTIFACT];                                       // the -9999 branch is a constant
  for (int c = 0; c < N_DEPTH_BINS * N_TYPES; ++c) sink(slot + c, c == cell ? wa * ga : 0.f);
  slot += N_DEPTH_BINS * N_TYPES;
  for (int c = 0; c < N_DEPTH_BINS * N_TYPES; ++c) sink(slot + c, c == cell ? wa * gb : 0.f);
  slot += N_DEPTH_BINS * N_TYPES;
  const float wn = r[NORMAL_ARTIFACT], wn2 = R.nalt < 1.f ? 0.f : wn;
  beta_binomial_grads(R.ndepth, R.nalt, S.na_alpha[ncell], S.na_beta[ncell], ga, gb);
  for (int c = 0; c < N_DEPTH_BINS * N_TYPES; ++c) sink(slot + c, c == ncell ? wn2 * ga : 0.f);
  slot += N_DEPTH_BINS * N_TYPES;
  for (int c = 0; c < N_DEPTH_BINS * N_TYPES; ++c) sink(slot + c, c == ncell ? wn2 * gb : 0.f);
  slot += N_DEPTH_BINS * N_TYPES;
  beta_binomial_grads(R.depth, R.alt, I.a_b, I.b_b, ga, gb);
  const float unclamped = (I.conc - I.a_b) > 0.001f ? 1.f : 0.f, mult = S.na_mult[vt];
  const float d_mult = ga * I.naf * I.conc - gb * unclamped * I.naf * I.conc;
  const float d_conc = ga * I.naf * mult + gb * unclamped * (1.f - I.naf * mult);
  for (int t = 0; t < N_TYPES; ++t) sink(slot + t, t == vt ? wn * d_mult : 0.f);
  slot += N_TYPES;
  for (int t = 0; t < N_TYPES; ++t) sink(slot + t, t == vt ? wn * d_conc : 0.f);
  slot += N_TYPES;
  for (int t = 0; t < N_TYPES; ++t)
#pragma unroll
    for (int c = 0; c < N_CALLS; ++c) sink(slot + t * N_CALLS + c, t == vt ? r[c] : 0.f);
}

template <bool FIT>
__global__ void __launch_bounds__(THREADS)
log_posteriors_kernel(const PmtPosteriorDesc D, const float* __restrict__ P, const int16_t* __restrict__ ints, long long int_stride,
                      const void* __restrict__ floats, int float_kind, long long float_stride, int n_variants,
                      PmtPosteriorOutputs out, FitArgs fit) {
  __shared__ float sp[small_count(PMT_POSTERIOR_MAX_COMPONENTS)];
  const int K = D.n_components;
  const int n_small = small_count(K);
  for (int i = threadIdx.x; i < n_small; i += blockDim.x) sp[i] = P[i];
  __syncthreads();
  const Spectra S = spectra_view(sp, K);
  const float* snv_rrra = P + n_small;   // [5][5][5][5], global (L1 / L2)

  extern __shared__ float wsum[];   // FIT: [WARPS][slot_count]
  const int n_slots = slot_count(K);
  if (FIT) {
    for (int i = threadIdx.x; i < WARPS * n_slots; i += blockDim.x) wsum[i] = 0.f;
    __syncthreads();
  }
  const int v_raw = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = v_raw < n_variants;
  if (!FIT && !valid) return;
  const int v = valid ? v_raw : n_variants - 1;     // FIT: out-of-range threads take part in the reductions with weight 0
  const Record R = load_record(ints, int_stride, floats, float_kind, float_stride, v);

  float pri[N_CALLS], spec[N_CALLS], norm[N_CALLS], post[N_CALLS];
  float mix_term[FIT ? MAXK : 1], mix_dcf[FIT ? MAXK : 1];
  Ingredients I;
  record_tables<FIT>(D, S, snv_rrra, R, 0, 1, NoMerge{}, (float*)mix_term, (float*)mix_dcf, pri, spec, norm, post, I);

  const long long o = (long long)v * N_CALLS;
#pragma unroll
  for (int c = 0; c < N_CALLS; ++c) {
    if (out.log_priors_bc) out.log_priors_bc[o + c] = pri[c];
    if (out.spectra_log_lks_bc) out.spectra_log_lks_bc[o + c] = spec[c];
    if (out.normal_log_lks_bc) out.normal_log_lks_bc[o + c] = norm[c];
    if (out.log_posteriors_bc) out.log_posteriors_bc[o + c] = post[c];
  }
  if (FIT) {
    // ---- E step + gradient of -mean log evidence (posterior_model.py:139-151) ----
    float r[N_CALLS];
    evidence_terms(S, K, R, I, (float*)mix_term, (float*)mix_dcf, post, valid ? 1.f : 0.f, r,
                   [&](int slot, float val) { slot_add(wsum, n_slots, slot, val); });
    if (valid && R.vt == 0 && (fit.somatic_snv_totals_rrra || fit.snv_context_totals_rrra)) {
      const int at = snv_context_cell(D, R.ir);
      if (fit.somatic_snv_totals_rrra) atomicAdd(fit.somatic_snv_totals_rrra + at, r[SOMATIC]);
      if (fit.snv_context_totals_rrra) atomicAdd(fit.snv_context_totals_rrra + at, 1.f);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_slots; i += blockDim.x) {
      float t = 0.f;
#pragma unroll
      for (int wq = 0; wq < WARPS; ++wq) t += wsum[wq * n_slots + i];
      fit.partials[(long long)blockIdx.x * n_slots + i] = t;
    }
    if (!valid) return;
  }
  if (out.posterior_probabilities_bc) {
    float m = post[0];
#pragma unroll
    for (int c = 1; c < N_CALLS; ++c) m = fmaxf(m, post[c]);
    float e[N_CALLS], s = 0.f;
#pragma unroll
    for (int c = 0; c < N_CALLS; ++c) { e[c] = expf(post[c] - m); s += e[c]; }
#pragma unroll
    for (int c = 0; c < N_CALLS; ++c) out.posterior_probabilities_bc[o + c] = e[c] / s;
  }
}

// Sums the per-CTA slots in CTA order (bitwise reproducible) and applies -1/B to the loss and gradient slots.
__global__ void fit_reduce_kernel(const float* __restrict__ partials, int n_blocks, int n_slots, int n_grad_slots, float inv_b,
                                  float* __restrict__ loss_out, float* __restrict__ grads_out, float* __restrict__ totals_tc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_slots) return;
  float s = 0.f;
  for (int b = 0; b < n_blocks; ++b) s += partials[(long long)b * n_slots + i];
  if (i == 0) { if (loss_out) *loss_out = -s * inv_b; }
  else if (i <= n_grad_slots) { if (grads_out) grads_out[i - 1] = -s * inv_b; }
  else if (totals_tc) totals_tc[i - 1 - n_grad_slots] += s;
}


// ---- one pass of the fit (learn_priors_and_spectra's batch loop, posterior_model.py:128-151) on a cluster of CTAs ------
// A warp per record: lane l takes the interpolation points j = l, l + 32, ... of every mixture component and the warp
// merges the 32 streaming states; the rest of the record's math runs on every lane (identical values).  A record's slot
// terms go to a row of shared memory; the rows are summed slot by slot in record order, so the pass is bitwise
// reproducible without atomics.  A cluster of C CTAs (ranks) takes a batch's records in chunks of up to C * PASS_ROWS,
// rank r a contiguous range of at most PASS_ROWS of them in its own shared memory.  Every rank then sums every rank's
// rows, in rank order through distributed shared memory, and runs the VJP and Adam itself: the sums see the rows in
// record order whatever C is, so each rank holds the bits of the one-CTA pass (C = 1) and no second exchange of the
// results is needed.  Rank 0 alone writes to global memory.
constexpr int PASS_WARPS = 16, PASS_THREADS = PASS_WARPS * 32, PASS_ROWS = 64;
constexpr int MAX_CLUSTER = 16;
constexpr int CONTEXT_CELLS = 625;
static_assert(PASS_THREADS >= 1 + 2 * MAXK + 4 * N_DEPTH_BINS * N_TYPES + 2 * N_TYPES + N_TYPES * N_CALLS, "a thread per slot");
static_assert(2 * PASS_THREADS >= CONTEXT_CELLS, "two context cells per thread");

struct FitPassArgs {
  PmtPosteriorDesc D;
  const float* params;             // constrained values of the raw parameters at the start, priors (constant in a pass)
  float* raw;                      // [2K + 70] raw spectra entries, grads_out order (in / out)
  float* adam_m;                   // [2K + 70] (in / out)
  float* adam_v;                   // [2K + 70] (in / out)
  long long* adam_step;            // [1] Adam steps taken so far (in / out)
  double lr;
  const int16_t* ints;
  long long int_stride;
  const void* floats;
  int float_kind;
  long long float_stride;
  long long n_records;
  int batch_size, n_batches;
  float* batch_losses;             // [n_batches]
  float* totals_tc;                // [5][5] +=, may be null
  float* somatic_snv_totals_rrra;  // [625] +=, may be null
  float* snv_context_totals_rrra;  // [625] +=, may be null
  float* context_ws;               // [2][625] the pass's context totals (workspace)
};

// OnlineD of the whole warp; the combination is symmetric in its two operands (no FMA contraction), so every lane ends
// with the same bits
__device__ __forceinline__ OnlineD warp_merge(OnlineD u) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, u.m, o), s2 = __shfl_xor_sync(0xffffffffu, u.s, o),
                d2 = __shfl_xor_sync(0xffffffffu, u.d, o);
    const float m = fmaxf(u.m, m2);
    const float a = u.m == m ? 1.f : expf(u.m - m), b = m2 == m ? 1.f : expf(m2 - m);
    u.s = __fadd_rn(__fmul_rn(u.s, a), __fmul_rn(s2, b));
    u.d = __fadd_rn(__fmul_rn(u.d, a), __fmul_rn(d2, b));
    u.m = m;
  }
  return u;
}
struct WarpMerge {
  __device__ __forceinline__ OnlineD operator()(const OnlineD& u) const { return warp_merge(u); }
};
// A lane's own [MAXK] array in a warp's [MAXK][32] block of shared memory (entry k of every lane in another bank)
struct LaneMix {
  float* p;
  __device__ __forceinline__ float& operator[](int k) const { return p[k * 32]; }
};

// One problem's pass on the calling cluster (a lone CTA: C = 1); smem: fit_pass_smem(K) bytes or more per CTA
__device__ __forceinline__ void fit_pass(const FitPassArgs& A, float* smem) {
  namespace cg = cooperative_groups;
  const cg::cluster_group cluster = cg::this_cluster();
  const int n_ranks = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  const bool lead = rank == 0;
  // C = 1 keeps the CTA barrier; a cluster barrier also orders the ranks' shared-memory writes before the others' reads
  auto pass_sync = [&]() {
    if (n_ranks == 1) __syncthreads();
    else cluster.sync();
  };
  const PmtPosteriorDesc& D = A.D;
  const int K = D.n_components, n_small = small_count(K), n_slots = slot_count(K), n_grad = n_slots - 1 - N_TYPES * N_CALLS;
  const int row_w = n_slots + 2;                 // slots, then the record's context cell (-1: none) and SOMATIC posterior
  float* sp = smem;                              // [n_small] constrained parameters of the current step
  float* gsh = sp + small_count(MAXK);           // [2K + 70] gradient, then raw values, of the current step
  float* mix = gsh + 2 * MAXK + 70;              // [PASS_WARPS][2][MAXK][32] per lane: responsibilities, mean d/d cf_k
  float* rows = mix + PASS_WARPS * 2 * MAXK * 32;   // [PASS_ROWS][row_w]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < n_small; i += PASS_THREADS) sp[i] = A.params[i];
  const float* snv_rrra = A.params + n_small;
  // a thread per raw entry (grads_out order; constrained index i, or i + 4 past the four fixed background entries)
  float raw = 0.f, m1 = 0.f, m2 = 0.f;
  const int si = tid < 2 * K ? tid : tid + 4;
  if (tid < n_grad) { raw = A.raw[tid]; m1 = A.adam_m[tid]; m2 = A.adam_v[tid]; }
  const long long step0 = *A.adam_step;
  const bool row_cells = A.somatic_snv_totals_rrra || A.snv_context_totals_rrra;   // rows carry their context cells
  const bool context = lead && row_cells;        // rank 0 keeps the context totals
  // context cells c0 = tid and c1 = tid + PASS_THREADS are this thread's, for the whole pass
  const int c0 = tid, c1 = tid + PASS_THREADS;
  if (context) {
    if (c0 < CONTEXT_CELLS) { A.context_ws[c0] = 0.f; A.context_ws[CONTEXT_CELLS + c0] = 0.f; }
    if (c1 < CONTEXT_CELLS) { A.context_ws[c1] = 0.f; A.context_ws[CONTEXT_CELLS + c1] = 0.f; }
  }
  float pass_total = 0.f;                        // thread 1 + n_grad + t: posterior_totals_tc slot t over the pass
  __syncthreads();
  const Spectra S = spectra_view(sp, K);
  const LaneMix mix_term{mix + warp * 2 * MAXK * 32 + lane}, mix_dcf{mix_term.p + MAXK * 32};

  for (int b = 0; b < A.n_batches; ++b) {
    const long long r0 = (long long)b * A.batch_size;
    const int nb = (int)min((long long)A.batch_size, A.n_records - r0);
    float acc = 0.f;                             // thread s < n_slots: slot s summed over the batch
    for (int q0 = 0; q0 < nb; q0 += n_ranks * PASS_ROWS) {
      const int nq = min(n_ranks * PASS_ROWS, nb - q0);
      const int per = (nq + n_ranks - 1) / n_ranks;   // rank r's records: [r * per, (r + 1) * per) of the chunk's nq
      const int lo = min(nq, rank * per), hi = min(nq, lo + per);
      float ctx[4] = {0.f, 0.f, 0.f, 0.f};        // the context cells' running values (hidden behind the E step)
      if (context) {
        if (c0 < CONTEXT_CELLS) { ctx[0] = A.context_ws[c0]; ctx[1] = A.context_ws[CONTEXT_CELLS + c0]; }
        if (c1 < CONTEXT_CELLS) { ctx[2] = A.context_ws[c1]; ctx[3] = A.context_ws[CONTEXT_CELLS + c1]; }
      }
      for (int q = lo + warp; q < hi; q += PASS_WARPS) {
        const Record R = load_record(A.ints, A.int_stride, A.floats, A.float_kind, A.float_stride, r0 + q0 + q);
        float pri[N_CALLS], spec[N_CALLS], norm[N_CALLS], post[N_CALLS], r[N_CALLS];
        Ingredients I;
        record_tables<true>(D, S, snv_rrra, R, lane, 32, WarpMerge{}, mix_term, mix_dcf, pri, spec, norm, post, I);
        float* row = rows + (q - lo) * row_w;
        evidence_terms(S, K, R, I, mix_term, mix_dcf, post, 1.f, r, [&](int slot, float val) {
          if ((slot & 31) == lane) row[slot] = val;
        });
        if (lane == 0) {
          row[n_slots] = __int_as_float(row_cells && R.vt == 0 ? snv_context_cell(D, R.ir) : -1);
          row[n_slots + 1] = r[SOMATIC];
        }
      }
      pass_sync();
      // the rows of n records from `src`, next in record order
      bool hit0 = false, hit1 = false;
      auto take_rows = [&](const float* src, int n) {
        if (tid < n_slots)
          for (int q = 0; q < n; ++q) acc += src[q * row_w + tid];
        if (context)
          for (int q = 0; q < n; ++q) {
            const int cell = __float_as_int(src[q * row_w + n_slots]);
            if (cell == c0) { ctx[0] += src[q * row_w + n_slots + 1]; ctx[1] += 1.f; hit0 = true; }
            else if (cell == c1) { ctx[2] += src[q * row_w + n_slots + 1]; ctx[3] += 1.f; hit1 = true; }
          }
      };
      if (n_ranks == 1) take_rows(rows, nq);
      else
        for (int rr = 0; rr < n_ranks; ++rr) {
          const int rlo = min(nq, rr * per);
          take_rows(rr == rank ? rows : cluster.map_shared_rank(rows, rr), min(nq, rlo + per) - rlo);
        }
      if (hit0) { A.context_ws[c0] = ctx[0]; A.context_ws[CONTEXT_CELLS + c0] = ctx[1]; }
      if (hit1) { A.context_ws[c1] = ctx[2]; A.context_ws[CONTEXT_CELLS + c1] = ctx[3]; }
      pass_sync();                               // no rank overwrites its rows while another still reads them
    }
    // ---- loss and gradient w.r.t. the constrained spectra (fit_reduce_kernel's -1/B) ----
    const float inv_b = 1.f / (float)nb;
    if (tid == 0) { if (lead) A.batch_losses[b] = -acc * inv_b; }
    else if (tid <= n_grad) gsh[tid - 1] = -acc * inv_b;
    else if (tid < n_slots) pass_total += acc;
    __syncthreads();
    // ---- vector-Jacobian product through the parametrisations, then Adam (torch.optim.Adam's defaults) ----
    if (tid < n_grad) {
      const float gw = gsh[tid], w = sp[si];
      float g;
      if (tid < K || (tid >= 2 * K + 4 * N_DEPTH_BINS * N_TYPES && tid < 2 * K + 4 * N_DEPTH_BINS * N_TYPES + N_TYPES)) {
        g = gw * (1.f - w) * w;                  // BoundedNumber(0, 1): sigmoid
      } else if (tid < 2 * K) {                  // LogWeights: log_softmax
        float sg = 0.f;
        for (int k = 0; k < K; ++k) sg += gsh[K + k];
        g = gw - expf(w) * sg;
      } else {
        g = gw * w;                              // PositiveNumber: exp
      }
      const long long t = step0 + b + 1;
      const double bc1 = 1.0 - pow(0.9, (double)t), bc2 = 1.0 - pow(0.999, (double)t);
      const float step_size = (float)(-(A.lr / bc1)), bc2_sqrt = (float)sqrt(bc2);
      m1 = m1 + 0.1f * (g - m1);
      m2 = m2 * 0.999f;
      m2 = m2 + 0.001f * g * g;
      const float denom = sqrtf(m2) / bc2_sqrt + 1e-8f;
      raw = raw + step_size * (m1 / denom);
    }
    __syncthreads();
    if (tid < n_grad) gsh[tid] = raw;
    __syncthreads();
    // ---- constrained values of the next step ----
    if (tid < n_grad) {
      float w;
      if (tid < K || (tid >= 2 * K + 4 * N_DEPTH_BINS * N_TYPES && tid < 2 * K + 4 * N_DEPTH_BINS * N_TYPES + N_TYPES)) {
        w = pmt::sigmoidf(raw);
      } else if (tid < 2 * K) {
        float mx = -INFINITY;
        for (int k = 0; k < K; ++k) mx = fmaxf(mx, gsh[K + k]);
        float se = 0.f;
        for (int k = 0; k < K; ++k) se += expf(gsh[K + k] - mx);
        w = (raw - mx) - logf(se);
      } else {
        w = expf(raw);
      }
      sp[si] = w;
    }
    __syncthreads();
  }
  // ---- the pass's results ----
  if (!lead) return;
  if (tid < n_grad) { A.raw[tid] = raw; A.adam_m[tid] = m1; A.adam_v[tid] = m2; }
  if (tid == 0) *A.adam_step = step0 + A.n_batches;
  if (A.totals_tc && tid > n_grad && tid < n_slots) A.totals_tc[tid - 1 - n_grad] += pass_total;
  if (context) {
    for (int c = tid; c < CONTEXT_CELLS; c += PASS_THREADS) {
      if (A.somatic_snv_totals_rrra) A.somatic_snv_totals_rrra[c] += A.context_ws[c];
      if (A.snv_context_totals_rrra) A.snv_context_totals_rrra[c] += A.context_ws[CONTEXT_CELLS + c];
    }
  }
}

__global__ void __launch_bounds__(PASS_THREADS, 1) fit_pass_kernel(const FitPassArgs A) {
  extern __shared__ float smem[];
  fit_pass(A, smem);
}

// A cluster per problem: every rank of cluster i copies problem i's arguments from a table in global memory to its shared
// memory first (the pass reads them throughout, and its own global writes would otherwise force re-loads)
__global__ void __launch_bounds__(PASS_THREADS, 1) fit_pass_many_kernel(const FitPassArgs* __restrict__ table) {
  extern __shared__ float smem[];
  __shared__ FitPassArgs A;
  static_assert(sizeof(FitPassArgs) % sizeof(int) == 0 && sizeof(FitPassArgs) / sizeof(int) <= PASS_THREADS, "a word per thread");
  const unsigned problem = blockIdx.x / cooperative_groups::this_cluster().num_blocks();
  if (threadIdx.x < sizeof(FitPassArgs) / sizeof(int))
    reinterpret_cast<int*>(&A)[threadIdx.x] = reinterpret_cast<const int*>(table + problem)[threadIdx.x];
  __syncthreads();
  fit_pass(A, smem);
}

size_t fit_pass_smem(int K) {
  return (size_t)(small_count(MAXK) + 2 * MAXK + 70 + PASS_WARPS * 2 * MAXK * 32 + PASS_ROWS * (slot_count(K) + 2)) * sizeof(float);
}

}  // namespace post

extern "C" int pmt_posterior_param_count(int32_t n_components) {
  return 2 * n_components + 4 + 4 * post::N_DEPTH_BINS * post::N_TYPES + 2 * post::N_TYPES + post::N_TYPES * post::N_CALLS + 625;
}

extern "C" int pmt_posterior_log_posteriors(const PmtPosteriorDesc* desc, const float* params, const int16_t* int_array,
                                            int64_t int_stride, const void* float_array, int32_t float_kind, int64_t float_stride,
                                            int32_t n_variants, const PmtPosteriorOutputs* out, void* stream) {
  PMT_CHECK(desc && params && int_array && float_array && out, "pmt_posterior_log_posteriors: null argument");
  PMT_CHECK(desc->n_components >= 1 && desc->n_components <= PMT_POSTERIOR_MAX_COMPONENTS, "somatic spectrum components %d outside 1..%d",
            desc->n_components, PMT_POSTERIOR_MAX_COMPONENTS);
  PMT_CHECK(float_kind == PMT_F16 || float_kind == PMT_F32, "float_kind must be PMT_F16 or PMT_F32");
  PMT_CHECK(!desc->use_context_dependent_snv_priors || desc->hap_len >= 3, "context-dependent SNV priors need haplotypes of >= 3 bases");
  if (n_variants <= 0) return 0;
  const int threads = 128, blocks = (n_variants + threads - 1) / threads;
  post::log_posteriors_kernel<false><<<blocks, threads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      *desc, params, int_array, int_stride, float_array, float_kind, float_stride, n_variants, *out, post::FitArgs{});
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_posterior_log_posteriors launch failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" size_t pmt_posterior_fit_workspace_size(int32_t n_variants, int32_t n_components) {
  const size_t blocks = (size_t)(n_variants + post::THREADS - 1) / post::THREADS;
  return blocks * post::slot_count(n_components) * sizeof(float) + 256;
}

extern "C" int pmt_posterior_fit_step(const PmtPosteriorDesc* desc, const float* params, const int16_t* int_array,
                                      int64_t int_stride, const void* float_array, int32_t float_kind, int64_t float_stride,
                                      int32_t n_variants, float* loss_out, float* grads_out, float* posterior_totals_tc,
                                      float* somatic_snv_totals_rrra, float* snv_context_totals_rrra, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  PMT_CHECK(desc && params && int_array && float_array && workspace, "pmt_posterior_fit_step: null argument");
  PMT_CHECK(desc->n_components >= 1 && desc->n_components <= PMT_POSTERIOR_MAX_COMPONENTS, "somatic spectrum components %d outside 1..%d",
            desc->n_components, PMT_POSTERIOR_MAX_COMPONENTS);
  PMT_CHECK(float_kind == PMT_F16 || float_kind == PMT_F32, "float_kind must be PMT_F16 or PMT_F32");
  PMT_CHECK(n_variants > 0, "empty batch");
  PMT_CHECK(workspace_bytes >= pmt_posterior_fit_workspace_size(n_variants, desc->n_components), "workspace too small");
  PMT_CHECK((!somatic_snv_totals_rrra && !snv_context_totals_rrra) || desc->hap_len >= 3, "SNV context totals need haplotypes of >= 3 bases");
  PMT_CHECK(!desc->use_context_dependent_snv_priors || desc->hap_len >= 3, "context-dependent SNV priors need haplotypes of >= 3 bases");
  const int K = desc->n_components, n_slots = post::slot_count(K), blocks = (n_variants + post::THREADS - 1) / post::THREADS;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  post::FitArgs fit{reinterpret_cast<float*>(workspace), somatic_snv_totals_rrra, snv_context_totals_rrra};
  PmtPosteriorOutputs none{};
  const size_t smem = (size_t)post::WARPS * n_slots * sizeof(float);
  post::log_posteriors_kernel<true><<<blocks, post::THREADS, smem, st>>>(*desc, params, int_array, int_stride, float_array, float_kind,
                                                                         float_stride, n_variants, none, fit);
  const int n_grad = 2 * K + 4 * post::N_DEPTH_BINS * post::N_TYPES + 2 * post::N_TYPES;
  post::fit_reduce_kernel<<<(n_slots + 127) / 128, 128, 0, st>>>(fit.partials, blocks, n_slots, n_grad, 1.f / (float)n_variants, loss_out,
                                                                grads_out, posterior_totals_tc);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_posterior_fit_step launch failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" size_t pmt_posterior_fit_pass_workspace_size(int32_t n_components) {
  if (n_components < 1 || n_components > PMT_POSTERIOR_MAX_COMPONENTS) return 0;
  return 2 * post::CONTEXT_CELLS * sizeof(float) + 256;
}

// The refusals of one fit-pass problem (`who` names the call, and the problem of a many-launch); on success *out holds
// the kernel's arguments with context_ws as the problem's context scratch
static int fit_pass_args(const PmtPosteriorFitProblem& p, const char* who, float* context_ws, post::FitPassArgs* out) {
  const PmtPosteriorDesc& d = p.desc;
  PMT_CHECK(p.params && p.raw_params && p.adam_m && p.adam_v && p.adam_step && p.int_array && p.float_array && p.batch_losses_out,
            "%s: null argument", who);
  PMT_CHECK(d.n_components >= 1 && d.n_components <= PMT_POSTERIOR_MAX_COMPONENTS, "%s: somatic spectrum components %d outside 1..%d",
            who, d.n_components, PMT_POSTERIOR_MAX_COMPONENTS);
  PMT_CHECK(p.batch_size >= 1, "%s: batch_size %d < 1", who, p.batch_size);
  PMT_CHECK(p.float_kind == PMT_F16 || p.float_kind == PMT_F32, "%s: float_kind must be PMT_F16 or PMT_F32", who);
  PMT_CHECK(p.n_records > 0, "%s: no records", who);
  const int64_t n_batches = (p.n_records + p.batch_size - 1) / p.batch_size;
  PMT_CHECK(n_batches <= INT32_MAX, "%s: %lld batches exceed the int32 range", who, (long long)n_batches);
  PMT_CHECK((!p.somatic_snv_totals_rrra && !p.snv_context_totals_rrra) || d.hap_len >= 3,
            "%s: SNV context totals need haplotypes of >= 3 bases", who);
  PMT_CHECK(!d.use_context_dependent_snv_priors || d.hap_len >= 3, "%s: context-dependent SNV priors need haplotypes of >= 3 bases", who);
  *out = post::FitPassArgs{d, p.params, p.raw_params, p.adam_m, p.adam_v, reinterpret_cast<long long*>(p.adam_step), p.learning_rate,
                           p.int_array, p.int_stride, p.float_array, p.float_kind, p.float_stride, p.n_records, p.batch_size,
                           (int)n_batches, p.batch_losses_out, p.posterior_totals_tc, p.somatic_snv_totals_rrra,
                           p.snv_context_totals_rrra, context_ws};
  return 0;
}

// The cluster launch of a fit-pass kernel: n_clusters clusters of `ctas` CTAs; `attr` holds the cluster dimension
static cudaLaunchConfig_t fit_pass_config(int n_clusters, int ctas, size_t smem, cudaStream_t st, cudaLaunchAttribute* attr) {
  attr->id = cudaLaunchAttributeClusterDimension;
  attr->val.clusterDim.x = (unsigned)ctas;
  attr->val.clusterDim.y = attr->val.clusterDim.z = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(n_clusters * ctas));
  cfg.blockDim = dim3(post::PASS_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cfg;
}

// The cluster width C of a fit-pass launch of `kernel` (smem bytes of dynamic shared memory per CTA) over n_problems
// problems whose largest batch is max_batch records, into *ctas; sets the kernel attributes the launch needs.
// PMT_POSTERIOR_CTAS when set, otherwise the largest C of 16, 8, 4 and 2 such that
//   - C <= ceil(max_batch / 16): a rank gives each record a warp, and a rank with fewer records than warps idles;
//   - every problem's cluster is resident at once (cudaOccupancyMaxActiveClusters), so no cluster waits for a second wave;
//   - there are fewer problems than SMs: from there on one CTA per problem fills the GPU by itself;
// and C = 1 (a CTA per problem) when none is.
static int fit_pass_ctas(const void* kernel, int n_problems, long long max_batch, size_t smem, const char* who, int* ctas) {
  const int forced = pmt_posterior_ctas_override();
  PMT_CHECK(forced != 0, "%s: PMT_POSTERIOR_CTAS must be 1, 2, 4, 8 or 16", who);
  PMT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  PMT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  if (forced > 0) {
    *ctas = forced;
    return 0;
  }
  int dev = 0, n_sm = 0;
  PMT_CUDA(cudaGetDevice(&dev));
  PMT_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  *ctas = 1;
  if (n_problems >= n_sm) return 0;
  for (int c = post::MAX_CLUSTER; c > 1; c /= 2) {
    if (16LL * (c - 1) >= max_batch) continue;                     // c > ceil(max_batch / 16)
    cudaLaunchAttribute attr;
    const cudaLaunchConfig_t cfg = fit_pass_config(1, c, smem, nullptr, &attr);
    int resident = 0;
    PMT_CUDA(cudaOccupancyMaxActiveClusters(&resident, kernel, &cfg));
    if (n_problems <= resident) {
      *ctas = c;
      return 0;
    }
  }
  return 0;
}

extern "C" int pmt_posterior_fit_pass(const PmtPosteriorDesc* desc, const float* params, float* raw_params, float* adam_m, float* adam_v,
                                      int64_t* adam_step, double learning_rate, const int16_t* int_array, int64_t int_stride,
                                      const void* float_array, int32_t float_kind, int64_t float_stride, int64_t n_records,
                                      int32_t batch_size, float* batch_losses_out, float* posterior_totals_tc,
                                      float* somatic_snv_totals_rrra, float* snv_context_totals_rrra, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  PMT_CHECK(desc && workspace, "pmt_posterior_fit_pass: null argument");
  const PmtPosteriorFitProblem p{*desc, params, raw_params, adam_m, adam_v, adam_step, learning_rate, int_array, int_stride, float_array,
                                 float_kind, float_stride, n_records, batch_size, batch_losses_out, posterior_totals_tc,
                                 somatic_snv_totals_rrra, snv_context_totals_rrra};
  post::FitPassArgs A;
  if (fit_pass_args(p, "pmt_posterior_fit_pass", reinterpret_cast<float*>(workspace), &A)) return 1;
  PMT_CHECK(workspace_bytes >= pmt_posterior_fit_pass_workspace_size(desc->n_components), "workspace too small: %zu bytes, need %zu",
            workspace_bytes, pmt_posterior_fit_pass_workspace_size(desc->n_components));
  const size_t smem = post::fit_pass_smem(desc->n_components);
  int ctas = 1;
  if (fit_pass_ctas((const void*)post::fit_pass_kernel, 1, std::min<long long>(batch_size, n_records), smem, "pmt_posterior_fit_pass",
                    &ctas))
    return 1;
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = fit_pass_config(1, ctas, smem, reinterpret_cast<cudaStream_t>(stream), &attr);
  const cudaError_t e = cudaLaunchKernelEx(&cfg, post::fit_pass_kernel, A);
  PMT_CHECK(e == cudaSuccess, "pmt_posterior_fit_pass launch failed: %s", cudaGetErrorString(e));
  return 0;
}

// Workspace of a many-launch: the device copy of the problem table (256-byte aligned), then [n_problems][2][625] floats
// of context scratch; the extra 256 bytes realign a caller's buffer
static size_t fit_pass_many_table_bytes(int32_t n_problems) {
  return ((size_t)n_problems * sizeof(post::FitPassArgs) + 255) & ~(size_t)255;
}

extern "C" size_t pmt_posterior_fit_pass_many_workspace_size(int32_t n_problems, int32_t max_components) {
  if (n_problems < 1 || max_components < 1 || max_components > PMT_POSTERIOR_MAX_COMPONENTS) return 0;
  return fit_pass_many_table_bytes(n_problems) + (size_t)n_problems * 2 * post::CONTEXT_CELLS * sizeof(float) + 256;
}

// The refusals of a many-launch's problems (`who` names the call); on success table[i] (when table is not null) holds
// problem i's kernel arguments with its share of context_ws, *max_k the largest K and *max_batch the largest batch
static int fit_pass_many_args(const PmtPosteriorFitProblem* h_problems, int32_t n_problems, const char* who, float* context_ws,
                              post::FitPassArgs* table, int* max_k, long long* max_batch) {
  PMT_CHECK(h_problems, "%s: null argument", who);
  PMT_CHECK(n_problems >= 1, "%s: n_problems %d < 1", who, n_problems);
  *max_k = 1;
  *max_batch = 1;
  for (int32_t i = 0; i < n_problems; ++i) {
    char problem[96];
    snprintf(problem, sizeof(problem), "%s: problem %d", who, i);
    post::FitPassArgs A;
    float* ws = context_ws ? context_ws + (size_t)i * 2 * post::CONTEXT_CELLS : nullptr;
    if (fit_pass_args(h_problems[i], problem, ws, table ? &table[i] : &A)) return 1;
    *max_k = std::max(*max_k, (int)h_problems[i].desc.n_components);
    *max_batch = std::max(*max_batch, std::min<long long>(h_problems[i].batch_size, h_problems[i].n_records));
  }
  return 0;
}

extern "C" int pmt_posterior_fit_ctas(const PmtPosteriorFitProblem* h_problems, int32_t n_problems) {
  const char* who = "pmt_posterior_fit_ctas";
  int max_k = 1, ctas = 0;
  long long max_batch = 1;
  if (fit_pass_many_args(h_problems, n_problems, who, nullptr, nullptr, &max_k, &max_batch)) return 0;
  // the kernel of the entry that would run these problems (both hold one CTA per SM)
  const void* kernel = n_problems == 1 ? (const void*)post::fit_pass_kernel : (const void*)post::fit_pass_many_kernel;
  if (fit_pass_ctas(kernel, n_problems, max_batch, post::fit_pass_smem(max_k), who, &ctas)) return 0;
  return ctas;
}

extern "C" int pmt_posterior_fit_pass_many(const PmtPosteriorFitProblem* h_problems, int32_t n_problems, void* workspace,
                                           size_t workspace_bytes, void* stream) {
  const char* who = "pmt_posterior_fit_pass_many";
  PMT_CHECK(h_problems && workspace, "%s: null argument", who);
  PMT_CHECK(n_problems >= 1, "%s: n_problems %d < 1", who, n_problems);
  unsigned char* base = pmt_align_up(workspace, 256);
  std::vector<post::FitPassArgs> table((size_t)n_problems);
  int max_k = 1;
  long long max_batch = 1;
  if (fit_pass_many_args(h_problems, n_problems, who, reinterpret_cast<float*>(base + fit_pass_many_table_bytes(n_problems)),
                         table.data(), &max_k, &max_batch))
    return 1;
  const size_t need = pmt_posterior_fit_pass_many_workspace_size(n_problems, max_k);
  PMT_CHECK(workspace_bytes >= need, "pmt_posterior_fit_pass_many: workspace too small: %zu bytes, need %zu", workspace_bytes, need);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  auto* d_table = reinterpret_cast<post::FitPassArgs*>(base);
  const size_t smem = post::fit_pass_smem(max_k);
  int ctas = 1;
  if (fit_pass_ctas((const void*)post::fit_pass_many_kernel, n_problems, max_batch, smem, who, &ctas)) return 1;
  // from pageable memory: the call returns once `table` has been staged, so it may go out of scope
  PMT_CUDA(cudaMemcpyAsync(d_table, table.data(), table.size() * sizeof(post::FitPassArgs), cudaMemcpyHostToDevice, st));
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = fit_pass_config(n_problems, ctas, smem, st, &attr);
  const cudaError_t e = cudaLaunchKernelEx(&cfg, post::fit_pass_many_kernel, (const post::FitPassArgs*)d_table);
  PMT_CHECK(e == cudaSuccess, "pmt_posterior_fit_pass_many launch failed: %s", cudaGetErrorString(e));
  return 0;
}
