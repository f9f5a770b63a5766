// Gradient of the clustering head, the rotation and the translation from the forward's per-read final features
// (sm_100a), without the trunk's backward.  pmt_head_backward serves steps in which nothing upstream of the rotation
// trains: the calibration epochs of model_training.py:145-147 and any fine-tuning of the head alone.
//
//   head_backward_kernel        CTA c takes a fixed run of variants, one warp per variant at a time; a warp splits into
//                               groups of LPR lanes (LPR = 8, 16 or 32 >= E), a group takes one read, lane e of the group
//                               holds feature e.  Gradients accumulate in lane-owned registers and per-group shared
//                               memory, are summed over groups and warps in a fixed order and land in CTA c's partial.
//   head_finish_kernel          sums the partials in CTA order, turns G = sum df f^T into dQ = G Q and D = sum df into
//                               dt = Q^T D (f = Q (y + t) with Q orthogonal, so y + t = Q^T f), writes the head's slots.
//
// The math is the head section of the FP32 backward (pmt_backward.cu, bwd_tail); the constants come from head_constants.
#include "pmt_call.h"
#include "pmt_host.h"
#include "pmt_tile.cuh"

namespace pmt {
namespace headbwd {

constexpr int THREADS = 512;
constexpr int WARPS = THREADS / 32;
constexpr int MAX_GROUPS = 4;                     // LPR >= 8
constexpr int MAX_ACC = PMT_MAX_FEAT * PMT_MAX_FEAT + 3 * PMT_MAX_FEAT + PMT_MAX_CLUSTERS * PMT_MAX_FEAT + 5 * PMT_MAX_CLUSTERS;
constexpr unsigned FULL = 0xffffffffu;

// Slots of one partial: [G: E*E][D: E][sigma: E][unit: K*E][tau, mu, emg sigma, lambda, log weight: K each]
struct Acc {
  int G, D, sigma, unit, scal, n;
};
__host__ __device__ inline Acc acc_layout(int E, int K) {
  Acc a;
  a.G = 0; a.D = E * E; a.sigma = a.D + E; a.unit = a.sigma + E; a.scal = a.unit + K * E; a.n = a.scal + 5 * K;
  return a;
}
__host__ __device__ inline int lanes_per_read(int E) { return E <= 8 ? 8 : (E <= 16 ? 16 : 32); }

__device__ __forceinline__ float group_sum(float x, int lpr) {
  for (int o = lpr >> 1; o > 0; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
  return x;
}
__device__ __forceinline__ float across_groups(float x, int lpr) {
  for (int o = lpr; o < 32; o <<= 1) x += __shfl_xor_sync(FULL, x, o);
  return x;
}

__global__ void __launch_bounds__(THREADS) head_backward_kernel(const PmtModelDesc D, const float* __restrict__ W,
                                                                 const int64_t* __restrict__ ref_off,
                                                                 const int64_t* __restrict__ alt_off, int B,
                                                                 const float* __restrict__ final_re,
                                                                 const float* __restrict__ d_logits_bk,
                                                                 const float* __restrict__ d_alt_means,
                                                                 const float* __restrict__ d_ref_means, int per_cta,
                                                                 float* __restrict__ partials) {
  __shared__ HeadConst HC;
  __shared__ float us[PMT_MAX_CLUSTERS * PMT_MAX_FEAT];
  __shared__ float scal[WARPS][MAX_GROUPS][5 * PMT_MAX_CLUSTERS];   // per-cluster scalars, one row per read group
  __shared__ float cta[MAX_ACC];
  const int E = D.d_feat, K = D.n_clusters;
  const Acc AL = acc_layout(E, K);
  const int lpr = lanes_per_read(E), ng = 32 / lpr;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane / lpr, e = lane % lpr;
  const bool fe = e < E;
  if (threadIdx.x == 0) head_constants(D, W, &HC);
  for (int i = threadIdx.x; i < K * E; i += THREADS) us[i] = W[D.unit_ke + i];
  for (int i = threadIdx.x; i < WARPS * MAX_GROUPS * 5 * PMT_MAX_CLUSTERS; i += THREADS) (&scal[0][0][0])[i] = 0.f;
  __syncthreads();
  float* my_scal = scal[warp][grp];
  const float s = fe ? HC.sigma[e] : 1.f;
  const long long total_ref = __ldg(ref_off + B);

  float a_sigma = 0.f, a_D = 0.f, a_unit[PMT_MAX_CLUSTERS], a_G[PMT_MAX_FEAT];
#pragma unroll
  for (int k = 0; k < PMT_MAX_CLUSTERS; ++k) a_unit[k] = 0.f;
#pragma unroll
  for (int j = 0; j < PMT_MAX_FEAT; ++j) a_G[j] = 0.f;

  const int v_lo = blockIdx.x * per_cta, v_hi = min(B, v_lo + per_cta);
  for (int v = v_lo + warp; v < v_hi; v += WARPS) {
    const long long r0 = __ldg(ref_off + v), r1 = __ldg(ref_off + v + 1);
    const long long a0 = __ldg(alt_off + v), a1 = __ldg(alt_off + v + 1);
    const long long nref = r1 - r0, nalt = a1 - a0;
    const float* gv = d_logits_bk ? d_logits_bk + (long long)v * (K + 2) : nullptr;
    const float g0 = gv ? __ldg(gv) : 0.f, g1 = gv ? __ldg(gv + 1) : 0.f;
    const float d_alt = (fe && d_alt_means) ? __ldg(d_alt_means + (long long)v * E + e) / ((float)nalt + 1e-4f) : 0.f;
    // ref rows enter only through the ref mean: sum df f^T over them is d_ref (sum f)^T
    if (d_ref_means) {
      float sf = 0.f;
      for (long long i = grp; i < nref; i += ng) sf += fe ? __ldg(final_re + (r0 + i) * E + e) : 0.f;
      sf = across_groups(sf, lpr);
      const float d_ref = fe ? __ldg(d_ref_means + (long long)v * E + e) / ((float)nref + 1e-4f) : 0.f;
      const float dr = grp == 0 ? d_ref : 0.f;     // every group holds the sum; group 0 adds it
      a_D = fmaf(dr, (float)nref, a_D);
#pragma unroll
      for (int j = 0; j < PMT_MAX_FEAT; ++j)
        if (j < E) a_G[j] = fmaf(dr, __shfl_sync(FULL, sf, j, lpr), a_G[j]);
    }
    // the log cluster weight enters each variant's logit once (feature_clustering.py:115-116)
    if (lane == 0 && gv)
      for (int k = 0; k < K; ++k) my_scal[4 * K + k] += __ldg(gv + 2 + k);
    for (long long base = 0; base < nalt; base += ng) {
      const bool live = base + grp < nalt;
      const float f = (live && fe) ? __ldg(final_re + (total_ref + a0 + base + grp) * E + e) : 0.f;
      const float h0 = live ? g0 : 0.f, h1 = live ? g1 : 0.f;
      float df = -h0 * f / (s * s) - h1 * f / (4.f * s * s);
      if (fe) a_sigma += h0 * (-1.f / s + f * f / (s * s * s)) + h1 * (-1.f / s + f * f / (4.f * s * s * s));
#pragma unroll
      for (int k = 0; k < PMT_MAX_CLUSTERS; ++k) {
        if (k < K) {
          const float u = fe ? us[k * E + e] : 0.f;
          const float gk = (live && gv) ? __ldg(gv + 2 + k) : 0.f;
          const float p = group_sum(f * u, lpr);
          const float o = f - p * u;
          const float o2 = group_sum(o * o, lpr), odu = group_sum(o * u, lpr);
          const float tau = __ldg(W + D.tau_k + k), lam = __ldg(W + D.lambda_k + k), sg = __ldg(W + D.emg_sigma_k + k),
                      mu = __ldg(W + D.mu_k + k);
          const float zarg = (HC.shift[k] - p) / HC.sqrt2_sigma[k];
          const float dlp = dlogerfc(zarg);
          const float dpar_dp = -dlp / HC.sqrt2_sigma[k] - lam;
          const float c_orth = -1.f / HC.two_tau2[k];
          df += gk * (c_orth * (2.f * o - 2.f * odu * u) + dpar_dp * u);
          a_unit[k] += gk * (c_orth * (-2.f * f * odu - 2.f * p * o) + dpar_dp * f);
          if (e == 0) {
            my_scal[0 * K + k] += gk * (-(E - 1) / tau + o2 / (tau * tau * tau));
            my_scal[1 * K + k] += gk * (dlp / HC.sqrt2_sigma[k] + lam);
            my_scal[2 * K + k] += gk * (dlp * (1.41421356237f * lam - zarg / sg) + lam * lam * sg);
            my_scal[3 * K + k] += gk * (1.f / lam + dlp * sg * 0.70710678118f + mu + lam * sg * sg - p);
          }
        }
      }
      df = (live && fe) ? df + d_alt : 0.f;
      a_D += df;
#pragma unroll
      for (int j = 0; j < PMT_MAX_FEAT; ++j)
        if (j < E) a_G[j] = fmaf(df, __shfl_sync(FULL, f, j, lpr), a_G[j]);
    }
  }

  // groups -> lane e of group 0, then warps in order -> the CTA's partial
  a_sigma = across_groups(a_sigma, lpr);
  a_D = across_groups(a_D, lpr);
#pragma unroll
  for (int k = 0; k < PMT_MAX_CLUSTERS; ++k) a_unit[k] = across_groups(a_unit[k], lpr);
#pragma unroll
  for (int j = 0; j < PMT_MAX_FEAT; ++j) a_G[j] = across_groups(a_G[j], lpr);
  for (int w = 0; w < WARPS; ++w) {
    if (warp == w && lane < lpr && fe) {
      const bool first = w == 0;
      cta[AL.sigma + e] = first ? a_sigma : cta[AL.sigma + e] + a_sigma;
      cta[AL.D + e] = first ? a_D : cta[AL.D + e] + a_D;
#pragma unroll
      for (int k = 0; k < PMT_MAX_CLUSTERS; ++k)
        if (k < K) cta[AL.unit + k * E + e] = first ? a_unit[k] : cta[AL.unit + k * E + e] + a_unit[k];
#pragma unroll
      for (int j = 0; j < PMT_MAX_FEAT; ++j)
        if (j < E) cta[AL.G + e * E + j] = first ? a_G[j] : cta[AL.G + e * E + j] + a_G[j];
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < 5 * K; i += THREADS) {
    float t = 0.f;
    for (int w = 0; w < WARPS; ++w)
      for (int g = 0; g < ng; ++g) t += scal[w][g][i];
    cta[AL.scal + i] = t;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < AL.n; i += THREADS) partials[(long long)blockIdx.x * AL.n + i] = cta[i];
}

// Sums the partials in CTA order and writes the head's slots of d_weights (the rest was zeroed before).
__global__ void __launch_bounds__(256) head_finish_kernel(const PmtModelDesc D, const float* __restrict__ W,
                                                          const float* __restrict__ partials, int n_cta,
                                                          float* __restrict__ d_weights) {
  __shared__ float red[MAX_ACC];
  const int E = D.d_feat, K = D.n_clusters;
  const Acc AL = acc_layout(E, K);
  for (int i = threadIdx.x; i < AL.n; i += blockDim.x) {
    float t = 0.f;
    for (int c = 0; c < n_cta; ++c) t += partials[(long long)c * AL.n + i];
    red[i] = t;
  }
  __syncthreads();
  const float* Q = W + D.rotation;
  for (int idx = threadIdx.x; idx < E * E; idx += blockDim.x) {      // dQ = G Q
    const int i = idx / E, j = idx % E;
    float t = 0.f;
    for (int m = 0; m < E; ++m) t = fmaf(red[AL.G + i * E + m], Q[m * E + j], t);
    d_weights[D.rotation + idx] = t;
  }
  for (int j = threadIdx.x; j < E; j += blockDim.x) {                // dt = Q^T D
    float t = 0.f;
    for (int i = 0; i < E; ++i) t = fmaf(Q[i * E + j], red[AL.D + i], t);
    d_weights[D.translation + j] = t;
    d_weights[D.sigma_e + j] = red[AL.sigma + j];
  }
  for (int i = threadIdx.x; i < K * E; i += blockDim.x) d_weights[D.unit_ke + i] = red[AL.unit + i];
  const int offs[5] = {D.tau_k, D.mu_k, D.emg_sigma_k, D.lambda_k, D.logw_k};
  for (int i = threadIdx.x; i < 5 * K; i += blockDim.x) d_weights[offs[i / K] + i % K] = red[AL.scal + i];
}

}  // namespace headbwd
}  // namespace pmt

using namespace pmt;

static size_t head_partials_bytes(const PmtModelDesc* desc) {
  return (size_t)PMT_PARTIAL_CTAS * headbwd::acc_layout(desc->d_feat, desc->n_clusters).n * sizeof(float);
}

extern "C" size_t pmt_head_backward_workspace_size(const PmtModelDesc* desc) {
  Plan P;
  if (!desc || pmt_build_plan(desc, &P)) return 0;
  return head_partials_bytes(desc) + 256;
}

extern "C" int pmt_head_backward(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const float* final_re,
                                 const PmtOutGrads* grads, float* d_weights, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  PMT_CHECK(desc && batch, "pmt_head_backward: NULL descriptor or batch");
  Plan P;
  if (pmt_build_plan(desc, &P)) return 1;
  const size_t need = head_partials_bytes(desc) + 256;
  PMT_CHECK(workspace && workspace_bytes >= need, "workspace too small: %zu < %zu", workspace_bytes, need);
  PMT_CHECK(final_re, "pmt_head_backward needs the forward's per-read final features (final_re is NULL)");
  PMT_CHECK(batch->n_variants > 0, "empty batch");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int B = batch->n_variants;
  int grid = (B + headbwd::WARPS - 1) / headbwd::WARPS;
  if (grid > PMT_PARTIAL_CTAS) grid = PMT_PARTIAL_CTAS;
  const int per_cta = (B + grid - 1) / grid;
  grid = (B + per_cta - 1) / per_cta;
  float* partials = reinterpret_cast<float*>(pmt_align_up(workspace, 256));
  PMT_CUDA(cudaMemsetAsync(d_weights, 0, (size_t)desc->n_params * sizeof(float), st));
  headbwd::head_backward_kernel<<<grid, headbwd::THREADS, 0, st>>>(
      *desc, weights, batch->ref_off, batch->alt_off, B, final_re, grads ? grads->d_logits_bk : nullptr,
      grads ? grads->d_alt_means_be : nullptr, grads ? grads->d_ref_means_be : nullptr, per_cta, partials);
  headbwd::head_finish_kernel<<<1, 256, 0, st>>>(*desc, weights, partials, grid, d_weights);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_head_backward launch failed: %s", cudaGetErrorString(e));
  return 0;
}
