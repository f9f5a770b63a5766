// Flat optimiser step: misc_utils.backpropagate's clip_grad_norm_(max_norm) + AdamW.step (misc_utils.py:125-129,
// model_training.py:68-72) over ONE flat fp32 parameter buffer, two launches, no host synchronisation.
//   1. grad_sqnorm_kernel: fixed-order partial sums of g^2 (one per CTA)
//   2. adamw_kernel: every CTA re-adds the partials in the same order (total norm), derives the clip coefficient
//      min(1, max_norm / (norm + 1e-6)) (torch.nn.utils.clip_grad_norm_) and applies decoupled weight decay, moment
//      updates and the bias-corrected step exactly as torch.optim.AdamW does (amsgrad off, maximize off).
// Entries whose mask is 0 (parameters without a gradient, e.g. frozen during a calibration epoch) are left untouched,
// as torch skips parameters whose .grad is None.
#include "pmt_host.h"

namespace pmt {
namespace optim {

constexpr int NORM_CTAS = 64;
constexpr int NT = 256;

__global__ void __launch_bounds__(NT) grad_sqnorm_kernel(const float* __restrict__ g, const float* __restrict__ mask, long long n,
                                                          float* __restrict__ partials) {
  __shared__ float red[NT];
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long lo = (long long)blockIdx.x * per, hi = lo + per < n ? lo + per : n;
  float s = 0.f;
  for (long long i = lo + threadIdx.x; i < hi; i += NT) {
    const float v = (mask && mask[i] == 0.f) ? 0.f : g[i];
    s = fmaf(v, v, s);
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = NT / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) partials[blockIdx.x] = red[0];
}

struct AdamArgs {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  const float* mask;
  const float* partials;
  float* total_norm_out;
  long long n;
  int* step_count;   // per-entry number of updates taken (torch keeps one step counter per parameter)
  float lr, beta1, beta2, eps, weight_decay, max_norm;
};

__global__ void __launch_bounds__(NT) adamw_kernel(const AdamArgs A) {
  float total = 0.f;
  for (int c = 0; c < NORM_CTAS; ++c) total += A.partials[c];     // same order in every CTA
  const float norm = sqrtf(total);
  float coef = 1.f;
  if (A.max_norm > 0.f) coef = fminf(A.max_norm / (norm + 1e-6f), 1.f);
  if (blockIdx.x == 0 && threadIdx.x == 0 && A.total_norm_out) *A.total_norm_out = norm;
  const double lb1 = log((double)A.beta1), lb2 = log((double)A.beta2);
  for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < A.n; i += (long long)gridDim.x * NT) {
    if (A.mask && A.mask[i] == 0.f) continue;
    const float g = A.grad[i] * coef;
    float p = A.param[i];
    p *= 1.f - A.lr * A.weight_decay;
    const float m = A.beta1 * A.exp_avg[i] + (1.f - A.beta1) * g;              // exp_avg.lerp_(grad, 1 - beta1)
    const float v = A.beta2 * A.exp_avg_sq[i] + (1.f - A.beta2) * g * g;
    A.exp_avg[i] = m;
    A.exp_avg_sq[i] = v;
    const int t = ++A.step_count[i];
    const float bias1 = (float)(-expm1((double)t * lb1));                 // 1 - beta1^t
    const float bias2_sqrt = (float)sqrt(-expm1((double)t * lb2));        // sqrt(1 - beta2^t)
    const float denom = sqrtf(v) / bias2_sqrt + A.eps;
    A.param[i] = p - (A.lr / bias1) * (m / denom);
  }
}

}  // namespace optim
}  // namespace pmt

using namespace pmt::optim;

extern "C" size_t pmt_adamw_workspace_size(void) { return NORM_CTAS * sizeof(float) + 256; }

extern "C" int pmt_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int32_t* step_count,
                              const float* mask, int64_t n, float lr, float beta1, float beta2, float eps, float weight_decay, float max_norm,
                              float* total_norm_out, void* workspace, size_t workspace_bytes, void* stream) {
  PMT_CHECK(params && grads && exp_avg && exp_avg_sq && step_count && n > 0, "pmt_adamw_step: bad arguments");
  PMT_CHECK(workspace && workspace_bytes >= pmt_adamw_workspace_size(), "pmt_adamw_step: workspace too small");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  float* partials = reinterpret_cast<float*>(pmt_align_up(workspace, 256));
  grad_sqnorm_kernel<<<NORM_CTAS, NT, 0, st>>>(grads, mask, n, partials);
  AdamArgs A;
  A.param = params; A.grad = grads; A.exp_avg = exp_avg; A.exp_avg_sq = exp_avg_sq; A.mask = mask; A.partials = partials;
  A.total_norm_out = total_norm_out; A.n = n;
  A.lr = lr; A.beta1 = beta1; A.beta2 = beta2; A.eps = eps; A.weight_decay = weight_decay; A.max_norm = max_norm;
  A.step_count = step_count;
  int grid = (int)((n + NT - 1) / NT);
  if (grid > 148 * 8) grid = 148 * 8;
  adamw_kernel<<<grid, NT, 0, st>>>(A);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_adamw_step launch failed: %s", cudaGetErrorString(e));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Rotation matrix of torch's orthogonal parametrisation (matrix-exponential map, square weight;
// torch/nn/utils/parametrizations.py:_Orthogonal.forward as used by euclidean_transformation.py:11-14):
//   A = tril(X) - tril(X)^T,  Q = base @ exp(A).
// exp by scaling and squaring with fixed parameters in double (Taylor degree 14 of A / 2^6, six squarings), the same
// recipe as engine/plan.py:_orthogonal_without_sync, which needs ~45 tensor ops forward and ~90 backward on the host
// side of every training step.  One CTA, one thread per matrix element; the backward kernel recomputes the forward
// intermediates in shared memory and walks them in reverse.
// ------------------------------------------------------------------------------------------------
namespace expm {

constexpr int DEG = 14, SQ = 6, MAXN = 16;

// C = A @ B (n x n, row-major, shared memory); every thread (i, j) of the n x n grid computes one element
__device__ __forceinline__ double mm(const double* A, const double* B, int n, int i, int j) {
  double s = 0.0;
  for (int k = 0; k < n; ++k) s = fma(A[i * n + k], B[k * n + j], s);
  return s;
}
__device__ __forceinline__ double mm_nt(const double* A, const double* B, int n, int i, int j) {   // A @ B^T
  double s = 0.0;
  for (int k = 0; k < n; ++k) s = fma(A[i * n + k], B[j * n + k], s);
  return s;
}
__device__ __forceinline__ double mm_tn(const double* A, const double* B, int n, int i, int j) {   // A^T @ B
  double s = 0.0;
  for (int k = 0; k < n; ++k) s = fma(A[k * n + i], B[k * n + j], s);
  return s;
}

// Fills Bm (= A / 2^SQ) and the DEG + SQ + 1 intermediates: T[0..DEG-1] = Horner iterates (T[0] = I + B/DEG, T[m] for
// k = DEG-m), T[DEG-1] = Taylor polynomial, T[DEG-1+s] after s squarings.  Caller syncs afterwards.
__device__ void forward_chain(const float* __restrict__ X, int n, double* Bm, double* T, int i, int j, bool active) {
  const int nn = n * n;
  if (active) {
    const double xl_ij = j <= i ? (double)X[i * n + j] : 0.0, xl_ji = i <= j ? (double)X[j * n + i] : 0.0;
    Bm[i * n + j] = (xl_ij - xl_ji) * (1.0 / (double)(1 << SQ));
  }
  __syncthreads();
  if (active) T[i * n + j] = (i == j ? 1.0 : 0.0) + Bm[i * n + j] / (double)DEG;
  __syncthreads();
  for (int m = 1; m < DEG; ++m) {          // k = DEG - m
    if (active) T[m * nn + i * n + j] = (i == j ? 1.0 : 0.0) + mm(Bm, T + (m - 1) * nn, n, i, j) / (double)(DEG - m);
    __syncthreads();
  }
  for (int s = 0; s < SQ; ++s) {
    const double* S = T + (DEG - 1 + s) * nn;
    if (active) T[(DEG + s) * nn + i * n + j] = mm(S, S, n, i, j);
    __syncthreads();
  }
}

__global__ void forward_kernel(const float* __restrict__ X, const float* __restrict__ base, int n, float* __restrict__ Q) {
  extern __shared__ double sm[];
  const int nn = n * n, i = threadIdx.x / n, j = threadIdx.x % n;
  const bool active = threadIdx.x < nn;
  double* Bm = sm;
  double* T = sm + nn;
  forward_chain(X, n, Bm, T, i, j, active);
  const double* E = T + (DEG - 1 + SQ) * nn;
  if (active) {
    double q = E[i * n + j];
    if (base) {
      q = 0.0;
      for (int k = 0; k < n; ++k) q = fma((double)base[i * n + k], E[k * n + j], q);
    }
    Q[i * n + j] = (float)q;
  }
}

__global__ void backward_kernel(const float* __restrict__ X, const float* __restrict__ base, const float* __restrict__ dQ, int n,
                                float* __restrict__ dX) {
  extern __shared__ double sm[];
  const int nn = n * n, i = threadIdx.x / n, j = threadIdx.x % n;
  const bool active = threadIdx.x < nn;
  double* Bm = sm;
  double* T = sm + nn;
  double* G = T + (DEG + SQ) * nn;     // running gradient
  double* G2 = G + nn;
  double* dB = G2 + nn;
  forward_chain(X, n, Bm, T, i, j, active);
  if (active) {
    double g = (double)dQ[i * n + j];
    if (base) {                          // Q = base @ E  ->  dE = base^T @ dQ
      g = 0.0;
      for (int k = 0; k < n; ++k) g = fma((double)base[k * n + i], (double)dQ[k * n + j], g);
    }
    G[i * n + j] = g;
    dB[i * n + j] = 0.0;
  }
  __syncthreads();
  for (int s = SQ - 1; s >= 0; --s) {    // S' = S @ S  ->  dS = dS' @ S^T + S^T @ dS'
    const double* S = T + (DEG - 1 + s) * nn;
    if (active) G2[i * n + j] = mm_nt(G, S, n, i, j) + mm_tn(S, G, n, i, j);
    __syncthreads();
    double* t = G; G = G2; G2 = t;
  }
  for (int m = DEG - 1; m >= 1; --m) {   // T[m] = I + (B @ T[m-1]) / k,  k = DEG - m
    const double inv_k = 1.0 / (double)(DEG - m);
    if (active) {
      dB[i * n + j] += mm_nt(G, T + (m - 1) * nn, n, i, j) * inv_k;
      G2[i * n + j] = mm_tn(Bm, G, n, i, j) * inv_k;
    }
    __syncthreads();
    double* t = G; G = G2; G2 = t;
  }
  if (active) dB[i * n + j] += G[i * n + j] / (double)DEG;     // T[0] = I + B / DEG
  __syncthreads();
  if (active) {                          // B = (Xl - Xl^T) / 2^SQ, Xl = tril(X)
    const double d = (dB[i * n + j] - dB[j * n + i]) * (1.0 / (double)(1 << SQ));
    dX[i * n + j] = j <= i ? (float)d : 0.f;
  }
}

}  // namespace expm

extern "C" int pmt_orthogonal_forward(const float* x, const float* base, int32_t n, float* q, void* stream) {
  PMT_CHECK(x && q && n >= 1 && n <= expm::MAXN, "pmt_orthogonal_forward: n must be in 1..%d", expm::MAXN);
  const size_t smem = (size_t)(1 + expm::DEG + expm::SQ) * n * n * sizeof(double);
  expm::forward_kernel<<<1, ((n * n + 31) / 32) * 32, smem, reinterpret_cast<cudaStream_t>(stream)>>>(x, base, n, q);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_orthogonal_forward launch failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int pmt_orthogonal_backward(const float* x, const float* base, const float* d_q, int32_t n, float* d_x, void* stream) {
  PMT_CHECK(x && d_q && d_x && n >= 1 && n <= expm::MAXN, "pmt_orthogonal_backward: n must be in 1..%d", expm::MAXN);
  const size_t smem = (size_t)(4 + expm::DEG + expm::SQ) * n * n * sizeof(double);
  if (smem > 48 * 1024)
    PMT_CUDA(cudaFuncSetAttribute(expm::backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  expm::backward_kernel<<<1, ((n * n + 31) / 32) * 32, smem, reinterpret_cast<cudaStream_t>(stream)>>>(x, base, d_q, n, d_x);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_orthogonal_backward launch failed: %s", cudaGetErrorString(e));
  return 0;
}

// ================================================================================================
// Constraint maps of the parametrised tensors on the flat parameter buffer (parameterizations.py: PositiveNumber,
// BoundedNumber, UnitVector, LogWeights) and their vector-Jacobian products: one launch each instead of ~20 / ~30 tensor
// ops per training step.  Every CTA copies its share of the unconstrained entries (mask 0); the groups are walked by the
// warps of CTA 0, one group per warp trip.
// ================================================================================================
namespace pmt {
namespace optim {

struct GroupDesc { int type, off, rows, cols; float a, b; };   // PMT_CONSTRAINT_*; a, b: BoundedNumber size and minimum

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

template <bool BACKWARD>
__global__ void constraints_kernel(const float* __restrict__ raw, const float* __restrict__ w_in, const float* __restrict__ d_w,
                                   const unsigned char* __restrict__ mask, long long n, const GroupDesc* __restrict__ groups, int n_groups,
                                   float* __restrict__ out) {
  // unconstrained entries: forward w = raw, backward g = d_w
  const float* src = BACKWARD ? d_w : raw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    if (!mask[i]) out[i] = src[i];
  if (blockIdx.x != 0) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  for (int gi = warp; gi < n_groups; gi += n_warps) {
    const GroupDesc G = groups[gi];
    if (G.type == PMT_CONSTRAINT_EXP) {                    // PositiveNumber: exp(x)
      for (int i = lane; i < G.rows * G.cols; i += 32) {
        const int p = G.off + i;
        out[p] = BACKWARD ? d_w[p] * w_in[p] : expf(raw[p]);
      }
    } else if (G.type == PMT_CONSTRAINT_BOUNDED) {         // BoundedNumber: size * sigmoid(x) + min
      for (int i = lane; i < G.rows * G.cols; i += 32) {
        const int p = G.off + i;
        const float sg = 1.f / (1.f + expf(-raw[p]));
        out[p] = BACKWARD ? d_w[p] * G.a * sg * (1.f - sg) : fmaf(G.a, sg, G.b);
      }
    } else if (G.type == PMT_CONSTRAINT_LOGSOFTMAX) {      // LogWeights: log_softmax over the whole tensor
      const int cnt = G.rows * G.cols;
      float mx = -INFINITY;
      for (int i = lane; i < cnt; i += 32) mx = fmaxf(mx, raw[G.off + i]);
      mx = warp_max(mx);
      float se = 0.f;
      for (int i = lane; i < cnt; i += 32) se += expf(raw[G.off + i] - mx);
      const float lse = mx + logf(warp_sum(se));
      if (!BACKWARD) {
        for (int i = lane; i < cnt; i += 32) out[G.off + i] = raw[G.off + i] - lse;
      } else {
        float sg = 0.f;
        for (int i = lane; i < cnt; i += 32) sg += d_w[G.off + i];
        sg = warp_sum(sg);
        for (int i = lane; i < cnt; i += 32) out[G.off + i] = d_w[G.off + i] - expf(raw[G.off + i] - lse) * sg;
      }
    } else {                                               // UnitVector rows x / |x| (TWICE: normalised once more, quirk Q5)
      const bool twice = G.type == PMT_CONSTRAINT_UNIT_TWICE;
      for (int r = 0; r < G.rows; ++r) {
        const int base = G.off + r * G.cols;
        float ss = 0.f;
        for (int c = lane; c < G.cols; c += 32) { const float x = raw[base + c]; ss = fmaf(x, x, ss); }
        const float n1 = sqrtf(warp_sum(ss));
        float n2 = 1.f;
        if (twice) {
          float s2 = 0.f;
          for (int c = lane; c < G.cols; c += 32) { const float u = raw[base + c] / n1; s2 = fmaf(u, u, s2); }
          n2 = sqrtf(warp_sum(s2));
        }
        if (!BACKWARD) {
          for (int c = lane; c < G.cols; c += 32) { const float u = raw[base + c] / n1; out[base + c] = twice ? u / n2 : u; }
        } else {
          // gu <- (gu - u2 (u2 . gu)) / n2 (when normalised twice), then gx = (gu - u (u . gu)) / n1
          float dot2 = 0.f;
          if (twice) {
            for (int c = lane; c < G.cols; c += 32) { const float u2 = raw[base + c] / n1 / n2; dot2 = fmaf(u2, d_w[base + c], dot2); }
            dot2 = warp_sum(dot2);
          }
          float dot1 = 0.f;
          for (int c = lane; c < G.cols; c += 32) {
            const float u = raw[base + c] / n1;
            const float gu = twice ? (d_w[base + c] - (u / n2) * dot2) / n2 : d_w[base + c];
            dot1 = fmaf(u, gu, dot1);
          }
          dot1 = warp_sum(dot1);
          for (int c = lane; c < G.cols; c += 32) {
            const float u = raw[base + c] / n1;
            const float gu = twice ? (d_w[base + c] - (u / n2) * dot2) / n2 : d_w[base + c];
            out[base + c] = (gu - u * dot1) / n1;
          }
        }
      }
    }
  }
}

}  // namespace optim
}  // namespace pmt

static int constraints_launch(bool backward, const float* raw, const float* w, const float* d_w, const uint8_t* mask, int64_t n,
                              const PmtConstraintGroup* groups, int32_t n_groups, float* out, void* stream) {
  static_assert(sizeof(PmtConstraintGroup) == sizeof(pmt::optim::GroupDesc), "PmtConstraintGroup layout");
  PMT_CHECK(raw && mask && out && n > 0 && (n_groups == 0 || groups), "pmt_constraints: missing arguments");
  PMT_CHECK(!backward || (w && d_w), "pmt_constraints_backward: missing arguments");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int grid = (int)((n + 4 * 256 - 1) / (4 * 256));
  if (grid > 148) grid = 148;
  if (grid < 1) grid = 1;
  const pmt::optim::GroupDesc* g = reinterpret_cast<const pmt::optim::GroupDesc*>(groups);
  if (backward) pmt::optim::constraints_kernel<true><<<grid, 256, 0, st>>>(raw, w, d_w, mask, n, g, n_groups, out);
  else pmt::optim::constraints_kernel<false><<<grid, 256, 0, st>>>(raw, nullptr, nullptr, mask, n, g, n_groups, out);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_constraints launch failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int pmt_constraints_forward(const float* raw, const uint8_t* mask, int64_t n, const PmtConstraintGroup* groups, int32_t n_groups,
                                       float* w, void* stream) {
  return constraints_launch(false, raw, nullptr, nullptr, mask, n, groups, n_groups, w, stream);
}
extern "C" int pmt_constraints_backward(const float* raw, const float* w, const float* d_w, const uint8_t* mask, int64_t n,
                                        const PmtConstraintGroup* groups, int32_t n_groups, float* g, void* stream) {
  return constraints_launch(true, raw, w, d_w, mask, n, groups, n_groups, g, stream);
}
