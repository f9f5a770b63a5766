// Fused loss head: ArtifactModel.compute_batch_losses (artifact_model.py:299-325) with the two adversarial heads
// (compute_alt_count_losses :276-279, compute_source_prediction_losses :267-274, gradient reversal
// gradient_reversal/functional.py:6-22) and its backward.
//
// One thread per variant.  The heads are MLP programs (mlp.py:25-76) at most 32 wide whose weights are staged in
// shared memory; the forward of a variant lives in that thread's local arrays.  Weight gradients are reductions over
// variants: each layer's (dL/dy, input) pairs of the CTA's 128 variants are staged variant-minor in shared memory and
// every thread owns a fixed set of (n, k) weight entries, which it sums over the 128 variants in order and adds to a
// shared accumulator.  Tiles are assigned to CTAs statically and the CTA-private accumulators are reduced in CTA order,
// so gradients are bitwise reproducible.
#include <cstring>

#include "pmt_host.h"

namespace pmt {
namespace loss {

constexpr int NT = 128;          // variants per tile = threads per CTA
constexpr int NTP = NT + 4;      // row stride of the staged (dL/dy, input) pairs: 16-byte rows that start 4 banks apart
constexpr int MAXW = PMT_MAX_HEAD_DIM;
constexpr int MAXOPS = PMT_MAX_MLP_OPS;

__device__ __forceinline__ float softplus(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }
// BCEWithLogitsLoss(reduction='none')
__device__ __forceinline__ float bce_logits(float x, float y) { return fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x))); }

struct HeadRange { int lo, hi; };   // flat-weight range [lo, hi) covering every parameter of a head

__device__ __forceinline__ HeadRange head_range(const PmtLinearOp* ops, int n) {
  HeadRange r{1 << 30, 0};
  for (int i = 0; i < n; ++i) {
    const PmtLinearOp& o = ops[i];
    r.lo = min(r.lo, min(o.w_off, o.b_off));
    r.hi = max(r.hi, max(o.w_off + o.in_dim * o.out_dim, o.b_off + o.out_dim));
    if (o.flags & PMT_OP_SKIP_END) { r.lo = min(r.lo, o.alpha_off); r.hi = max(r.hi, o.alpha_off + 1); }
  }
  if (n == 0) { r.lo = 0; r.hi = 0; }
  return r;
}

// y[n] = b[n] + sum_k W[n][k] h[k] for n < N: four outputs at a time (independent accumulators; h[k] is read once per four
// FMAs -- the per-thread vectors live in local memory because the programs are run-time data)
__device__ __forceinline__ void dense4(const float* __restrict__ w, const float* __restrict__ b, int N, int K, const float* h, float* y) {
  for (int n0 = 0; n0 < N; n0 += 4) {
    const int n1 = min(n0 + 1, N - 1), n2 = min(n0 + 2, N - 1), n3 = min(n0 + 3, N - 1);
    const float *w0 = w + n0 * K, *w1 = w + n1 * K, *w2 = w + n2 * K, *w3 = w + n3 * K;
    float a0 = b[n0], a1 = b[n1], a2 = b[n2], a3 = b[n3];
    for (int k = 0; k < K; ++k) {
      const float hk = h[k];
      a0 = fmaf(w0[k], hk, a0); a1 = fmaf(w1[k], hk, a1); a2 = fmaf(w2[k], hk, a2); a3 = fmaf(w3[k], hk, a3);
    }
    y[n0] = a0;
    if (n0 + 1 < N) y[n0 + 1] = a1;
    if (n0 + 2 < N) y[n0 + 2] = a2;
    if (n0 + 3 < N) y[n0 + 3] = a3;
  }
}

// Forward of an MLP program on one vector.  hin[i] = the vector fed to Linear i (after the block's leading SELU);
// xin[i] = the block input at a SKIP_BEGIN op.  Returns the output in `x` (width of the last op).
__device__ void mlp_forward(const PmtLinearOp* ops, int n_ops, const float* w /* smem, offset by -lo */, float* x,
                            float (*hin)[MAXW], float (*xin)[MAXW]) {
  float res[MAXW], h[MAXW], y[MAXW];
  for (int i = 0; i < n_ops; ++i) {
    const PmtLinearOp& o = ops[i];
    const int K = o.in_dim, N = o.out_dim;
    if (o.flags & PMT_OP_SKIP_BEGIN) {
      for (int k = 0; k < K; ++k) { res[k] = x[k]; if (xin) xin[i][k] = x[k]; h[k] = selu(x[k]); }
    } else {
      for (int k = 0; k < K; ++k) h[k] = x[k];
    }
    if (hin) for (int k = 0; k < K; ++k) hin[i][k] = h[k];
    dense4(w + o.w_off, w + o.b_off, N, K, h, y);
    if (o.flags & PMT_OP_SKIP_END) {
      const float alpha = w[o.alpha_off];
      for (int n = 0; n < N; ++n) x[n] = res[n] + alpha * y[n];
    } else if (o.flags & PMT_OP_POST_SELU) {
      for (int n = 0; n < N; ++n) x[n] = selu(y[n]);
    } else {
      for (int n = 0; n < N; ++n) x[n] = y[n];
    }
  }
}

struct LossArgs {
  PmtLossDesc d;
  PmtLossBatch b;
  const float* wflat;
};

__device__ __forceinline__ void load_variant(const LossArgs& A, int v, float& label, float& is_labeled, float& alt_target, int& source,
                                             float& w, float& sw) {
  const int16_t* row = A.b.int_array + (long long)v * A.b.int_stride;
  const int code = row[A.b.label_col];
  label = code == 0 ? 1.f : (code == 2 ? 0.5f : 0.f);     // batch.py:66-68 (Label.ARTIFACT = 0, UNLABELED = 2)
  is_labeled = code != 2 ? 1.f : 0.f;
  const float alt = A.b.alt_counts ? (float)A.b.alt_counts[v] : (float)row[A.b.alt_count_col];
  alt_target = alt / A.d.max_alt_count;
  source = row[A.b.source_col];
  w = A.b.weights_b ? A.b.weights_b[v] : 1.f;
  sw = A.b.source_weights_b ? A.b.source_weights_b[v] : 1.f;
}

__global__ void __launch_bounds__(NT) losses_forward_kernel(const __grid_constant__ LossArgs A, PmtLossOutputs out) {
  extern __shared__ __align__(16) float ws[];
  const PmtLossDesc& D = A.d;
  const HeadRange ra = head_range(D.alt_ops, D.n_alt_ops), rs = head_range(D.src_ops, D.n_src_ops);
  float* wa = ws;
  float* wsrc = ws + (ra.hi - ra.lo);
  for (int i = threadIdx.x; i < ra.hi - ra.lo; i += NT) wa[i] = A.wflat[ra.lo + i];
  for (int i = threadIdx.x; i < rs.hi - rs.lo; i += NT) wsrc[i] = A.wflat[rs.lo + i];
  __syncthreads();
  const int E = D.d_feat;
  for (int v = blockIdx.x * NT + threadIdx.x; v < A.b.n_variants; v += gridDim.x * NT) {
    float label, is_labeled, alt_target, w, sw;
    int source;
    load_variant(A, v, label, is_labeled, alt_target, source, w, sw);
    const float sup = is_labeled * bce_logits(A.b.logits_b[v], label);
    const float xo = fminf(A.b.outlier_logits_b[v], D.max_outlier_logit);
    const float unsup = (1.f - is_labeled) * bce_logits(xo, 0.f);
    float x[MAXW];
    for (int e = 0; e < E; ++e) x[e] = A.b.features_be[(long long)v * E + e];
    mlp_forward(D.alt_ops, D.n_alt_ops, wa - ra.lo, x, nullptr, nullptr);
    const float pred = sigmoidf(x[0]);
    const float altl = (pred - alt_target) * (pred - alt_target);
    float srcl = 0.f;
    if (D.n_src_ops > 0) {
      for (int e = 0; e < E; ++e) x[e] = A.b.features_be[(long long)v * E + e];
      mlp_forward(D.src_ops, D.n_src_ops, wsrc - rs.lo, x, nullptr, nullptr);
      float mx = -INFINITY, den = 0.f;
      for (int s = 0; s < D.n_sources; ++s) mx = fmaxf(mx, x[s]);
      for (int s = 0; s < D.n_sources; ++s) { x[s] = expf(x[s] - mx); den += x[s]; }
      for (int s = 0; s < D.n_sources; ++s) { const float dlt = x[s] / den - (s == source ? 1.f : 0.f); srcl = fmaf(dlt, dlt, srcl); }
    }
    if (out.supervised_b) out.supervised_b[v] = sup;
    if (out.unsupervised_b) out.unsupervised_b[v] = unsup;
    if (out.alt_count_b) out.alt_count_b[v] = altl;
    if (out.source_b) out.source_b[v] = srcl;
    if (out.total_b) out.total_b[v] = w * (sup + unsup + altl) + sw * srcl;
  }
}

// Backward of one head for the CTA's tile: every thread holds dL/d(output) of its variant in g[] (zero for idle
// threads).  On return g[] = dL/d(head input).  Weight gradients go to the shared accumulator `acc` (offset by -lo).
__device__ void mlp_backward_tile(const PmtLinearOp* ops, int n_ops, const float* w, float* acc, float* g, float (*hin)[MAXW],
                                  float (*xin)[MAXW], float* sD, float* sA) {
  const int t = threadIdx.x;
  float gres[MAXW], gy[MAXW], gin[MAXW];
  for (int i = n_ops - 1; i >= 0; --i) {
    const PmtLinearOp& o = ops[i];
    const int K = o.in_dim, N = o.out_dim;
    float gdot = 0.f;
    if (o.flags & PMT_OP_SKIP_END) {
      const float alpha = w[o.alpha_off];
      dense4(w + o.w_off, w + o.b_off, N, K, hin[i], gin);   // gin: scratch for the block's un-scaled output y
      for (int n = 0; n < N; ++n) {
        gres[n] = g[n];
        gdot = fmaf(g[n], gin[n], gdot);           // d alpha
        gy[n] = alpha * g[n];
      }
    } else if (o.flags & PMT_OP_POST_SELU) {
      // the activated output is what the next op consumed: its block input (SKIP_BEGIN) or its linear input
      const float* aout = (i + 1 < n_ops && (ops[i + 1].flags & PMT_OP_SKIP_BEGIN)) ? xin[i + 1] : hin[i + 1];
      for (int n = 0; n < N; ++n) gy[n] = g[n] * selu_grad_from_out(aout[n]);
    } else {
      for (int n = 0; n < N; ++n) gy[n] = g[n];
    }
    // ---- weight / bias / alpha gradients: stage (gy, hin) variant-minor, then each thread sums its (n, k) entries ----
    __syncthreads();
    for (int n = 0; n < N; ++n) sD[n * NTP + t] = gy[n];
    for (int k = 0; k < K; ++k) sA[k * NTP + t] = hin[i][k];
    sD[MAXW * NTP + t] = gdot;
    __syncthreads();
    // lanes of a warp read different rows k of sA (16 bytes each, rows 4 banks apart: conflict-free) and mostly one row n
    // of sD (broadcast); four partial sums, added in a fixed order
    for (int p = t; p < N * K; p += NT) {
      const int n = p / K, k = p - n * K;
      const float4* dr = reinterpret_cast<const float4*>(sD + n * NTP);
      const float4* ar = reinterpret_cast<const float4*>(sA + k * NTP);
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 4
      for (int r = 0; r < NT / 4; ++r) {
        const float4 dv = dr[r], av = ar[r];
        s0 = fmaf(dv.x, av.x, s0); s1 = fmaf(dv.y, av.y, s1); s2 = fmaf(dv.z, av.z, s2); s3 = fmaf(dv.w, av.w, s3);
      }
      acc[o.w_off + p] += (s0 + s1) + (s2 + s3);
    }
    if (t < N) {
      const float4* dr = reinterpret_cast<const float4*>(sD + t * NTP);
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      for (int r = 0; r < NT / 4; ++r) { const float4 dv = dr[r]; s0 += dv.x; s1 += dv.y; s2 += dv.z; s3 += dv.w; }
      acc[o.b_off + t] += (s0 + s1) + (s2 + s3);
    }
    if ((o.flags & PMT_OP_SKIP_END) && t == 32) {   // a lane of the second warp: the first one carries the bias sums too
      float s = 0.f;
      for (int r = 0; r < NT; ++r) s += sD[MAXW * NTP + r];
      acc[o.alpha_off] += s;
    }
    // ---- data gradient: four inputs k at a time ----
    for (int k0 = 0; k0 < K; k0 += 4) {
      const int k1 = min(k0 + 1, K - 1), k2 = min(k0 + 2, K - 1), k3 = min(k0 + 3, K - 1);
      const float* wr = w + o.w_off;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      for (int n = 0; n < N; ++n) {
        const float gn = gy[n];
        s0 = fmaf(wr[n * K + k0], gn, s0); s1 = fmaf(wr[n * K + k1], gn, s1); s2 = fmaf(wr[n * K + k2], gn, s2); s3 = fmaf(wr[n * K + k3], gn, s3);
      }
      gin[k0] = s0;
      if (k0 + 1 < K) gin[k0 + 1] = s1;
      if (k0 + 2 < K) gin[k0 + 2] = s2;
      if (k0 + 3 < K) gin[k0 + 3] = s3;
    }
    if (o.flags & PMT_OP_SKIP_BEGIN) {
      for (int k = 0; k < K; ++k) g[k] = gres[k] + gin[k] * selu_grad_from_out(hin[i][k]);   // hin = SELU(block input)
    } else {
      for (int k = 0; k < K; ++k) g[k] = gin[k];
    }
  }
}

struct LossBwdArgs {
  LossArgs a;
  PmtLossGrads g;
  float* d_logits_b;
  float* d_outlier_logits_b;
  float* d_features_be;
  float* partials;   // [grid][n_head] CTA-private head-weight gradients (alt range, then source range)
};

__global__ void __launch_bounds__(NT) losses_backward_kernel(const __grid_constant__ LossBwdArgs B) {
  extern __shared__ __align__(16) float ws[];
  const LossArgs& A = B.a;
  const PmtLossDesc& D = A.d;
  const HeadRange ra = head_range(D.alt_ops, D.n_alt_ops), rs = head_range(D.src_ops, D.n_src_ops);
  const int na = ra.hi - ra.lo, ns = rs.hi - rs.lo;
  float* wa = ws;
  float* wsrc = wa + na;
  float* acca = wsrc + ns;
  float* accs = acca + na;
  float* sD = ws + ((2 * (na + ns) + 3) & ~3);   // [MAXW + 1][NTP], 16-byte aligned
  float* sA = sD + (MAXW + 1) * NTP;     // [MAXW][NTP]
  const int t = threadIdx.x;
  for (int i = t; i < na; i += NT) { wa[i] = A.wflat[ra.lo + i]; acca[i] = 0.f; }
  for (int i = t; i < ns; i += NT) { wsrc[i] = A.wflat[rs.lo + i]; accs[i] = 0.f; }
  __syncthreads();
  const int E = D.d_feat;
  const int n_tiles = (A.b.n_variants + NT - 1) / NT;
  float hin[MAXOPS][MAXW], xin[MAXOPS][MAXW];
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int v = tile * NT + t;
    const bool on = v < A.b.n_variants;
    float label = 0.f, is_labeled = 0.f, alt_target = 0.f, w = 0.f, sw = 0.f;
    int source = 0;
    if (on) load_variant(A, v, label, is_labeled, alt_target, source, w, sw);
    // upstream gradients of the five per-variant loss vectors (artifact_model.py:320-325)
    const float gt = on && B.g.g_total_b ? B.g.g_total_b[v] : 0.f;
    const float g_sup = (on && B.g.g_supervised_b ? B.g.g_supervised_b[v] : 0.f) + gt * w;
    const float g_uns = (on && B.g.g_unsupervised_b ? B.g.g_unsupervised_b[v] : 0.f) + gt * w;
    const float g_alt = (on && B.g.g_alt_count_b ? B.g.g_alt_count_b[v] : 0.f) + gt * w;
    const float g_src = (on && B.g.g_source_b ? B.g.g_source_b[v] : 0.f) + gt * sw;
    float dfeat[MAXW];
    for (int e = 0; e < MAXW; ++e) dfeat[e] = 0.f;
    if (on) {
      const float xl = A.b.logits_b[v];
      if (B.d_logits_b) B.d_logits_b[v] = g_sup * is_labeled * (sigmoidf(xl) - label);
      const float xo = A.b.outlier_logits_b[v];
      const float pass = xo <= D.max_outlier_logit ? 1.f : 0.f;               // torch.clip passes gradient on [min, max]
      if (B.d_outlier_logits_b) B.d_outlier_logits_b[v] = g_uns * (1.f - is_labeled) * sigmoidf(fminf(xo, D.max_outlier_logit)) * pass;
    }
    float x[MAXW], g[MAXW];
    // ---- alt-count head ----
    {
      for (int e = 0; e < MAXW; ++e) { x[e] = (on && e < E) ? A.b.features_be[(long long)v * E + e] : 0.f; g[e] = 0.f; }
      mlp_forward(D.alt_ops, D.n_alt_ops, wa - ra.lo, x, hin, xin);
      const float pred = sigmoidf(x[0]);
      g[0] = on ? g_alt * 2.f * (pred - alt_target) * pred * (1.f - pred) : 0.f;
      mlp_backward_tile(D.alt_ops, D.n_alt_ops, wa - ra.lo, acca - ra.lo, g, hin, xin, sD, sA);
      for (int e = 0; e < E; ++e) dfeat[e] -= D.alt_reversal * g[e];          // gradient reversal
    }
    // ---- source head ----
    if (D.n_src_ops > 0) {
      for (int e = 0; e < MAXW; ++e) { x[e] = (on && e < E) ? A.b.features_be[(long long)v * E + e] : 0.f; g[e] = 0.f; }
      mlp_forward(D.src_ops, D.n_src_ops, wsrc - rs.lo, x, hin, xin);
      const int S = D.n_sources;
      float mx = -INFINITY, den = 0.f, pd = 0.f;
      for (int s = 0; s < S; ++s) mx = fmaxf(mx, x[s]);
      for (int s = 0; s < S; ++s) { x[s] = expf(x[s] - mx); den += x[s]; }
      for (int s = 0; s < S; ++s) {
        x[s] /= den;
        g[s] = 2.f * (x[s] - (s == source ? 1.f : 0.f));                       // d loss / d prob
        pd = fmaf(x[s], g[s], pd);
      }
      for (int s = 0; s < S; ++s) g[s] = on ? g_src * x[s] * (g[s] - pd) : 0.f; // softmax backward
      mlp_backward_tile(D.src_ops, D.n_src_ops, wsrc - rs.lo, accs - rs.lo, g, hin, xin, sD, sA);
      for (int e = 0; e < E; ++e) dfeat[e] -= D.src_reversal * g[e];
    }
    if (on && B.d_features_be)
      for (int e = 0; e < E; ++e) B.d_features_be[(long long)v * E + e] = dfeat[e];
  }
  __syncthreads();
  float* part = B.partials + (long long)blockIdx.x * (na + ns);
  for (int i = t; i < na; i += NT) part[i] = acca[i];
  for (int i = t; i < ns; i += NT) part[na + i] = accs[i];
}

// d_weights[lo + i] = sum over CTAs (in CTA order) of the partials; every other entry of d_weights is zero.
// The last layer of a DenseSkipBlock accumulated dW = alpha * (g x h) directly, so no fix-up pass is needed here.
__global__ void losses_reduce_kernel(const float* __restrict__ partials, int n_cta, int na, int ns, int lo_a, int lo_s, int n_params,
                                     float* __restrict__ d_weights) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_params) return;
  float s = 0.f;
  int idx = -1;
  if (p >= lo_a && p < lo_a + na) idx = p - lo_a;
  else if (p >= lo_s && p < lo_s + ns) idx = na + (p - lo_s);
  if (idx >= 0)
    for (int c = 0; c < n_cta; ++c) s += partials[(long long)c * (na + ns) + idx];
  d_weights[p] = s;
}

}  // namespace loss
}  // namespace pmt

using namespace pmt;
using namespace pmt::loss;

static int check_desc(const PmtLossDesc* d) {
  PMT_CHECK(d && d->d_feat >= 1 && d->d_feat <= MAXW, "loss head: feature dimension must be in [1, %d]", MAXW);
  PMT_CHECK(d->n_alt_ops >= 1 && d->n_alt_ops <= MAXOPS && d->n_src_ops >= 0 && d->n_src_ops <= MAXOPS, "loss head: bad op counts");
  PMT_CHECK(d->n_sources >= 1 && d->n_sources <= MAXW, "loss head: number of sources must be in [1, %d]", MAXW);
  for (int h = 0; h < 2; ++h) {
    const PmtLinearOp* ops = h ? d->src_ops : d->alt_ops;
    const int n = h ? d->n_src_ops : d->n_alt_ops;
    for (int i = 0; i < n; ++i)
      PMT_CHECK(ops[i].in_dim >= 1 && ops[i].in_dim <= MAXW && ops[i].out_dim >= 1 && ops[i].out_dim <= MAXW,
                "loss head: layer widths above %d are not supported", MAXW);
    if (n > 0) PMT_CHECK(ops[0].in_dim == d->d_feat && ops[n - 1].out_dim == (h ? d->n_sources : 1), "loss head: program shape mismatch");
  }
  return 0;
}

static HeadRange host_range(const PmtLinearOp* ops, int n) {
  HeadRange r{1 << 30, 0};
  for (int i = 0; i < n; ++i) {
    const PmtLinearOp& o = ops[i];
    const int lo = o.w_off < o.b_off ? o.w_off : o.b_off;
    int hi = o.w_off + o.in_dim * o.out_dim;
    if (o.b_off + o.out_dim > hi) hi = o.b_off + o.out_dim;
    if (lo < r.lo) r.lo = lo;
    if (hi > r.hi) r.hi = hi;
    if (o.flags & PMT_OP_SKIP_END) {
      if (o.alpha_off < r.lo) r.lo = o.alpha_off;
      if (o.alpha_off + 1 > r.hi) r.hi = o.alpha_off + 1;
    }
  }
  if (n == 0) { r.lo = 0; r.hi = 0; }
  return r;
}

static int loss_grid(int n_variants) {
  int grid = (n_variants + NT - 1) / NT;
  if (grid > 148 * 4) grid = 148 * 4;
  return grid < 1 ? 1 : grid;
}

extern "C" size_t pmt_losses_workspace_size(const PmtLossDesc* desc, int32_t n_variants) {
  if (!desc) return 0;
  const HeadRange ra = host_range(desc->alt_ops, desc->n_alt_ops), rs = host_range(desc->src_ops, desc->n_src_ops);
  return (size_t)loss_grid(n_variants) * (size_t)((ra.hi - ra.lo) + (rs.hi - rs.lo)) * sizeof(float) + 256;
}

extern "C" int pmt_losses_forward(const PmtLossDesc* desc, const float* weights, const PmtLossBatch* batch, const PmtLossOutputs* out,
                                  void* stream) {
  if (check_desc(desc)) return 1;
  PMT_CHECK(batch && batch->n_variants > 0 && batch->logits_b && batch->outlier_logits_b && batch->features_be && batch->int_array,
            "pmt_losses_forward: missing inputs");
  const HeadRange ra = host_range(desc->alt_ops, desc->n_alt_ops), rs = host_range(desc->src_ops, desc->n_src_ops);
  LossArgs A;
  A.d = *desc; A.b = *batch; A.wflat = weights;
  const size_t smem = (size_t)((ra.hi - ra.lo) + (rs.hi - rs.lo)) * sizeof(float);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  PMT_CUDA(cudaFuncSetAttribute(losses_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  losses_forward_kernel<<<loss_grid(batch->n_variants), NT, smem, st>>>(A, *out);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_losses_forward launch failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int pmt_losses_backward(const PmtLossDesc* desc, const float* weights, const PmtLossBatch* batch, const PmtLossGrads* grads,
                                   float* d_logits_b, float* d_outlier_logits_b, float* d_features_be, float* d_weights,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  if (check_desc(desc)) return 1;
  PMT_CHECK(batch && batch->n_variants > 0 && grads && d_weights, "pmt_losses_backward: missing arguments");
  PMT_CHECK(workspace && workspace_bytes >= pmt_losses_workspace_size(desc, batch->n_variants), "pmt_losses_backward: workspace too small");
  const HeadRange ra = host_range(desc->alt_ops, desc->n_alt_ops), rs = host_range(desc->src_ops, desc->n_src_ops);
  const int na = ra.hi - ra.lo, ns = rs.hi - rs.lo;
  LossBwdArgs B;
  B.a.d = *desc; B.a.b = *batch; B.a.wflat = weights;
  B.g = *grads;
  B.d_logits_b = d_logits_b; B.d_outlier_logits_b = d_outlier_logits_b; B.d_features_be = d_features_be;
  B.partials = reinterpret_cast<float*>(pmt_align_up(workspace, 256));
  const int grid = loss_grid(batch->n_variants);
  const size_t smem = (size_t)(2 * (na + ns) + 8 + (2 * MAXW + 1) * NTP) * sizeof(float);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  PMT_CUDA(cudaFuncSetAttribute(losses_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  losses_backward_kernel<<<grid, NT, smem, st>>>(B);
  losses_reduce_kernel<<<(desc->n_params + 255) / 256, 256, 0, st>>>(B.partials, grid, na, ns, ra.lo, rs.lo, desc->n_params, d_weights);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_losses_backward launch failed: %s", cudaGetErrorString(e));
  return 0;
}
