// The context-dependent SNV-prior fit of architecture/snv_context_priors.py (fit_mutation_rates_sc) on the device, float64
// throughout: one CTA per problem, every problem of a cohort in one launch.
//
// Each problem is the same method as the host fit: the same start (the smoothed maximum-likelihood mu, log_sigma = -2),
// the same sample-average ELBO over 64 fixed standard-normal draws, its gradient written out by hand, and the algorithm
// of torch.optim.LBFGS(lr=1, max_iter=300, max_eval=375, tolerance_grad=1e-9, tolerance_change=1e-12, history_size=100,
// line_search_fn="strong_wolfe") with its _strong_wolfe / _cubic_interpolate line search step for step; E_q[rate_sc] is
// the mean over 1000 fixed draws.  Both draw tables are inputs (the host's _sobol_normal tables), so both fits see the
// same draws.  Results agree with the host's to rounding: the sums here run in a different (fixed) order.
//
// Every reduction is a fixed-order block reduction and problems never communicate, so a problem's result is the same
// bits whatever else is in the launch.  Every thread keeps the optimiser's scalar state itself: the scalars come out of
// reductions that every thread reads whole, so all threads take the same branches.  Element j of every 388-vector is
// read and written by thread j % NT only, so elementwise updates need no barrier; the reductions and the objective have
// their own.  The L-BFGS history (2 x 100 x 388 doubles) lives in the caller's workspace, everything else in shared memory.
#include <cuda_runtime.h>
#include <math.h>

#include <cstdio>

#include "../../include/permutect_b200.h"
#include "pmt_host.h"

namespace ctxfit {

constexpr int S = 12, CX = 16, CELLS = S * CX;            // substitutions x flank pairs
constexpr int D = 3 + (S - 1) + S * (CX - 1);             // 194 unconstrained coordinates
constexpr int P = 2 * D;                                  // mu then log_sigma, the order of the host's LBFGS parameters
constexpr int ELBO_DRAWS = 64, MEAN_DRAWS = 1000;
constexpr int UNITS = ELBO_DRAWS * S;                     // (draw, substitution) rows of the binomial term
constexpr int HISTORY = 100, MAX_ITER = 300, MAX_EVAL = MAX_ITER * 5 / 4;
constexpr double TOL_GRAD = 1e-9, TOL_CHANGE = 1e-12, LS_TOL_CHANGE = 1e-9;   // _strong_wolfe keeps its own default
constexpr double C1 = 1e-4, C2 = 0.9, MAX_LOG_RATE = -1e-12;
constexpr int NT = 256, NWARPS = NT / 32;
constexpr size_t HISTORY_BYTES = (size_t)2 * HISTORY * P * sizeof(double);

struct Smem {
  double total[CELLS], snv[CELLS];
  double x[P], xt[P], g[P], prev_g[P], dir[P];            // point, trial point, flat_grad, prev_flat_grad, d
  double g_new[P], g_prev[P], bracket_g[2][P];            // the line search's gradients
  double sig[D];                                          // exp(log_sigma) of the point being evaluated
  double gz[ELBO_DRAWS * D];                              // d lp / d z per draw; rate_sc per mean draw at the end
  double log_r[ELBO_DRAWS], zr[ELBO_DRAWS], a_s[ELBO_DRAWS], a_c[ELBO_DRAWS], lp0[ELBO_DRAWS], sum_lts[ELBO_DRAWS];
  double log_ts[ELBO_DRAWS * S];
  double row_g[UNITS], row_l[UNITS], row_lp[UNITS];       // per (draw, s): sum of d lp / d log_rate, sum log_tsc, lp part
  double ro[HISTORY], al[HISTORY];
  double red[NWARPS];
  double f;
};

// digamma for x > 0: the recurrence up to x >= 10, then the asymptotic series (as torch's CPU digamma does)
__device__ __forceinline__ double digamma(double x) {
  double r = 0.0;
  while (x < 10.0) {
    r -= 1.0 / x;
    x += 1.0;
  }
  const double z = 1.0 / (x * x);
  const double series = z * (1.0 / 12 - z * (1.0 / 120 - z * (1.0 / 252 - z * (1.0 / 240 - z * (1.0 / 132 - z * (691.0 / 32760 - z / 12))))));
  return r + log(x) - 0.5 / x - series;
}

__device__ __forceinline__ double log_sigmoid(double x) { return fmin(x, 0.0) - log1p(exp(-fabs(x))); }   // torch's form
__device__ __forceinline__ double sigmoid(double x) { return 1.0 / (1.0 + exp(-x)); }
// Python's max(a, b) / min(a, b): the first argument unless the second compares greater / smaller
__device__ __forceinline__ double py_max(double a, double b) { return b > a ? b : a; }
__device__ __forceinline__ double py_min(double a, double b) { return b < a ? b : a; }
// p + t * d: the trial points of the line search and the step taken, one expression so both are the same bits
__device__ __forceinline__ double step_to(double p, double t, double d) { return __fma_rn(t, d, p); }

// Fixed-order block sum, its result in every thread: a warp butterfly, then the warp partials in warp order
__device__ __forceinline__ double block_sum(double v, double* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = red[0];
  for (int w = 1; w < NWARPS; ++w) s += red[w];
  __syncthreads();
  return s;
}

__device__ __forceinline__ double nan_max(double a, double b) { return (a > b || a != a) ? a : b; }

__device__ __forceinline__ double block_max(double v, double* red) {
  for (int o = 16; o; o >>= 1) v = nan_max(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double m = red[0];
  for (int w = 1; w < NWARPS; ++w) m = nan_max(m, red[w]);
  __syncthreads();
  return m;
}

__device__ __forceinline__ double dot(const double* a, const double* b, double* red) {
  double s = 0.0;
  for (int j = threadIdx.x; j < P; j += NT) s += a[j] * b[j];
  return block_sum(s, red);
}

__device__ __forceinline__ double abs_max(const double* a, double scale, double* red) {
  double m = 0.0;
  for (int j = threadIdx.x; j < P; j += NT) m = nan_max(m, fabs(a[j] * scale));
  return block_max(m, red);
}

// The per-draw scalars of _log_joint at z = p + sig * e (coordinates 0..13): log_r, the two concentrations and the
// substitution simplex (log_softmax of [z_s, -sum z_s]); with `prior`, also the lp terms that need no cell.
__device__ void draw_scalars(Smem& sm, const double* p, const double* e, int slot, bool prior) {
  double z[3 + S - 1];
  for (int j = 0; j < 3 + S - 1; ++j) z[j] = p[j] + sm.sig[j] * e[j];
  const double log_r = log_sigmoid(z[0]), log_1mr = log_sigmoid(-z[0]);
  double y[S], zsum = 0.0;
  for (int k = 0; k < S - 1; ++k) {
    y[k] = z[3 + k];
    zsum += z[3 + k];
  }
  y[S - 1] = -zsum;
  double m = y[0];
  for (int k = 1; k < S; ++k) m = fmax(m, y[k]);
  double se = 0.0;
  for (int k = 0; k < S; ++k) se += exp(y[k] - m);
  const double lse = log(se);
  double sum_lts = 0.0;
  for (int k = 0; k < S; ++k) {
    const double lt = y[k] - m - lse;
    sm.log_ts[slot * S + k] = lt;
    sum_lts += lt;
  }
  sm.log_r[slot] = log_r;
  if (!prior) return;
  const double a_s = exp(z[1]), a_c = exp(z[2]);
  double lp = log(1e6) + (1e6 - 1) * log_1mr + log_r + log_1mr;                 // overall_rate ~ Beta(1, 1e6), log-odds
  const double gamma_const = 4 * log(5.0) - log(6.0);                           // Gamma(4, rate 5) through log
  lp = lp + (gamma_const + 3 * z[1] - 5 * a_s + z[1]);
  lp = lp + (gamma_const + 3 * z[2] - 5 * a_c + z[2]);
  lp = lp + lgamma(S * a_s) - S * lgamma(a_s) + (a_s - 1) * sum_lts + (log((double)S) + sum_lts);
  lp = lp + S * (lgamma(CX * a_c) - CX * lgamma(a_c));
  sm.zr[slot] = z[0];
  sm.a_s[slot] = a_s;
  sm.a_c[slot] = a_c;
  sm.sum_lts[slot] = sum_lts;
  sm.lp0[slot] = lp;
}

// log_softmax of the context simplex of row s of a draw: [z_sc[s], -sum z_sc[s]] -> lx[16]
__device__ __forceinline__ void context_simplex(const Smem& sm, const double* p, const double* e, int s, double* lx) {
  const int base = 3 + (S - 1) + s * (CX - 1);
  double zsum = 0.0;
  for (int c = 0; c < CX - 1; ++c) {
    lx[c] = p[base + c] + sm.sig[base + c] * e[base + c];
    zsum += lx[c];
  }
  lx[CX - 1] = -zsum;
  double m = lx[0];
  for (int c = 1; c < CX; ++c) m = fmax(m, lx[c]);
  double se = 0.0;
  for (int c = 0; c < CX; ++c) se += exp(lx[c] - m);
  const double lse = log(se);
  for (int c = 0; c < CX; ++c) lx[c] = lx[c] - m - lse;
}

// The objective at p[P], -(mean_d lp(mu + exp(log_sigma) * eps_d) + sum log_sigma), returned in every thread; its
// gradient goes to grad[P].  Starts with a barrier, so p may have just been written elementwise.
__device__ double evaluate(Smem& sm, const double* p, double* grad, const double* __restrict__ eps) {
  const int tid = threadIdx.x;
  __syncthreads();
  for (int j = tid; j < D; j += NT) sm.sig[j] = exp(p[D + j]);
  __syncthreads();
  if (tid < ELBO_DRAWS) draw_scalars(sm, p, eps + (size_t)tid * D, tid, true);
  __syncthreads();
  // the binomial term and the context simplex, one (draw, substitution) row per unit
  for (int u = tid; u < UNITS; u += NT) {
    const int d = u / S, s = u % S;
    double lx[CX];
    context_simplex(sm, p, eps + (size_t)d * D, s, lx);
    const double base = sm.log_r[d] + log((double)(S * CX)) + sm.log_ts[d * S + s];
    const double a_c = sm.a_c[d];
    double lp = 0.0, sum_g = 0.0, sum_l = 0.0, gl[CX], sum_gl = 0.0;
    for (int c = 0; c < CX; ++c) {
      const double l = base + lx[c];
      const bool pass = l <= MAX_LOG_RATE;                  // clamp(max=): the gradient passes where l <= max
      const double lc = pass ? l : MAX_LOG_RATE;
      const double w = exp(lc);
      const double tot = sm.total[s * CX + c], k = sm.snv[s * CX + c];
      lp += k * lc + (tot - k) * log1p(-w);
      const double G = pass ? k - (tot - k) * (w / (1.0 - w)) : 0.0;
      sum_g += G;
      sum_l += lx[c];
      gl[c] = G + a_c;                                      // (a_c - 1) * sum log_tsc + the log-Jacobian's sum log_tsc
      sum_gl += gl[c];
    }
    sm.row_lp[u] = lp + (a_c - 1) * sum_l + (log((double)CX) + sum_l);
    sm.row_g[u] = sum_g;
    sm.row_l[u] = sum_l;
    // log_softmax backward, then y = [z, -sum z]
    double* gz = sm.gz + (size_t)d * D + 3 + (S - 1) + s * (CX - 1);
    const double dy_last = gl[CX - 1] - exp(lx[CX - 1]) * sum_gl;
    for (int c = 0; c < CX - 1; ++c) gz[c] = (gl[c] - exp(lx[c]) * sum_gl) - dy_last;
  }
  __syncthreads();
  if (tid < ELBO_DRAWS) {
    const int d = tid;
    double lp = sm.lp0[d], sum_g = 0.0, sum_l = 0.0, gts[S], sum_gts = 0.0;
    for (int s = 0; s < S; ++s) {
      lp += sm.row_lp[d * S + s];
      sum_g += sm.row_g[d * S + s];
      sum_l += sm.row_l[d * S + s];
      gts[s] = sm.a_s[d] + sm.row_g[d * S + s];
      sum_gts += gts[s];
    }
    double* gz = sm.gz + (size_t)d * D;
    const double dy_last = gts[S - 1] - exp(sm.log_ts[d * S + S - 1]) * sum_gts;
    for (int k = 0; k < S - 1; ++k) gz[3 + k] = (gts[k] - exp(sm.log_ts[d * S + k]) * sum_gts) - dy_last;
    const double zr = sm.zr[d], a_s = sm.a_s[d], a_c = sm.a_c[d];
    gz[0] = (sum_g + 1.0) * sigmoid(-zr) - 1e6 * sigmoid(zr);
    gz[1] = (4.0 - 5.0 * a_s) + a_s * (S * digamma(S * a_s) - S * digamma(a_s) + sm.sum_lts[d]);
    gz[2] = (4.0 - 5.0 * a_c) + a_c * (S * CX * (digamma(CX * a_c) - digamma(a_c)) + sum_l);
    sm.lp0[d] = lp;
  }
  __syncthreads();
  for (int j = tid; j < D; j += NT) {
    double sg = 0.0, sge = 0.0;
    for (int d = 0; d < ELBO_DRAWS; ++d) {
      const double v = sm.gz[(size_t)d * D + j];
      sg += v;
      sge += v * eps[(size_t)d * D + j];
    }
    grad[j] = -(sg / ELBO_DRAWS);
    grad[D + j] = -(sge / ELBO_DRAWS) * sm.sig[j] - 1.0;
  }
  if (tid == 0) {
    double lps = 0.0, lss = 0.0;
    for (int d = 0; d < ELBO_DRAWS; ++d) lps += sm.lp0[d];
    for (int j = 0; j < D; ++j) lss += p[D + j];
    sm.f = -(lps / ELBO_DRAWS + lss);
  }
  __syncthreads();
  return sm.f;
}

// torch.optim.lbfgs._cubic_interpolate; bounded when lo <= hi is given
__device__ double cubic_interpolate(double x1, double f1, double g1, double x2, double f2, double g2, bool bounded, double lo,
                                    double hi) {
  if (!bounded) {
    lo = x1 <= x2 ? x1 : x2;
    hi = x1 <= x2 ? x2 : x1;
  }
  const double d1 = g1 + g2 - 3 * (f1 - f2) / (x1 - x2);
  const double d2_square = d1 * d1 - g1 * g2;
  if (d2_square >= 0) {
    const double d2 = sqrt(d2_square);
    const double min_pos = x1 <= x2 ? x2 - (x2 - x1) * ((g2 + d2 - d1) / (g2 - g1 + 2 * d2))
                                    : x1 - (x1 - x2) * ((g1 + d2 - d1) / (g1 - g2 + 2 * d2));
    return py_min(py_max(min_pos, lo), hi);
  }
  return (lo + hi) / 2.0;
}

__device__ __forceinline__ void copy(double* dst, const double* src) {
  for (int j = threadIdx.x; j < P; j += NT) dst[j] = src[j];
}

// The objective and gradient at x + t d into g_new; returns f, *gtd = g_new . d
__device__ __forceinline__ double directional(Smem& sm, double t, const double* eps, double* gtd) {
  for (int j = threadIdx.x; j < P; j += NT) sm.xt[j] = step_to(sm.x[j], t, sm.dir[j]);
  const double f = evaluate(sm, sm.xt, sm.g_new, eps);
  *gtd = dot(sm.g_new, sm.dir, sm.red);
  return f;
}

// torch.optim.lbfgs._strong_wolfe from x along dir with the loss f, gradient sm.g and gtd; on return sm.g holds the
// gradient at the accepted step, *t the step, and the result is its loss.  *ls_evals counts the evaluations.
__device__ double strong_wolfe(Smem& sm, const double* eps, double* t_io, double f, double gtd, int max_ls, int* ls_evals) {
  double t = *t_io;
  const double d_norm = abs_max(sm.dir, 1.0, sm.red);
  double gtd_new;
  double f_new = directional(sm, t, eps, &gtd_new);
  int evals = 1;
  double t_prev = 0, f_prev = f, gtd_prev = gtd;
  copy(sm.g_prev, sm.g);
  bool done = false;
  int ls_iter = 0, n_bracket = 0;
  double br[2], br_f[2], br_gtd[2];
  while (ls_iter < max_ls) {
    if (f_new > (f + C1 * t * gtd) || (ls_iter > 1 && f_new >= f_prev)) {
      br[0] = t_prev; br[1] = t; br_f[0] = f_prev; br_f[1] = f_new; br_gtd[0] = gtd_prev; br_gtd[1] = gtd_new;
      copy(sm.bracket_g[0], sm.g_prev);
      copy(sm.bracket_g[1], sm.g_new);
      n_bracket = 2;
      break;
    }
    if (fabs(gtd_new) <= -C2 * gtd) {
      br[0] = br[1] = t; br_f[0] = br_f[1] = f_new;
      copy(sm.bracket_g[0], sm.g_new);
      n_bracket = 1;
      done = true;
      break;
    }
    if (gtd_new >= 0) {
      br[0] = t_prev; br[1] = t; br_f[0] = f_prev; br_f[1] = f_new; br_gtd[0] = gtd_prev; br_gtd[1] = gtd_new;
      copy(sm.bracket_g[0], sm.g_prev);
      copy(sm.bracket_g[1], sm.g_new);
      n_bracket = 2;
      break;
    }
    const double min_step = t + 0.01 * (t - t_prev), max_step = t * 10;
    const double tmp = t;
    t = cubic_interpolate(t_prev, f_prev, gtd_prev, t, f_new, gtd_new, true, min_step, max_step);
    t_prev = tmp;
    f_prev = f_new;
    copy(sm.g_prev, sm.g_new);
    gtd_prev = gtd_new;
    f_new = directional(sm, t, eps, &gtd_new);
    ++evals;
    ++ls_iter;
  }
  if (ls_iter == max_ls) {
    br[0] = 0; br[1] = t; br_f[0] = f; br_f[1] = f_new;
    copy(sm.bracket_g[0], sm.g);
    copy(sm.bracket_g[1], sm.g_new);
    n_bracket = 2;
  }
  // zoom
  bool insuf_progress = false;
  int low = br_f[0] <= br_f[n_bracket - 1] ? 0 : 1, high = 1 - low;
  while (!done && ls_iter < max_ls) {
    if (fabs(br[1] - br[0]) * d_norm < LS_TOL_CHANGE) break;
    t = cubic_interpolate(br[0], br_f[0], br_gtd[0], br[1], br_f[1], br_gtd[1], false, 0, 0);
    const double bmax = py_max(br[0], br[1]), bmin = py_min(br[0], br[1]);
    const double eps_b = 0.1 * (bmax - bmin);
    if (py_min(bmax - t, t - bmin) < eps_b) {
      if (insuf_progress || t >= bmax || t <= bmin) {
        t = fabs(t - bmax) < fabs(t - bmin) ? bmax - eps_b : bmin + eps_b;
        insuf_progress = false;
      } else {
        insuf_progress = true;
      }
    } else {
      insuf_progress = false;
    }
    f_new = directional(sm, t, eps, &gtd_new);
    ++evals;
    ++ls_iter;
    if (f_new > (f + C1 * t * gtd) || f_new >= br_f[low]) {
      br[high] = t; br_f[high] = f_new; br_gtd[high] = gtd_new;
      copy(sm.bracket_g[high], sm.g_new);
      low = br_f[0] <= br_f[1] ? 0 : 1;
      high = 1 - low;
    } else {
      if (fabs(gtd_new) <= -C2 * gtd) {
        done = true;
      } else if (gtd_new * (br[high] - br[low]) >= 0) {
        br[high] = br[low]; br_f[high] = br_f[low]; br_gtd[high] = br_gtd[low];
        copy(sm.bracket_g[high], sm.bracket_g[low]);
      }
      br[low] = t; br_f[low] = f_new; br_gtd[low] = gtd_new;
      copy(sm.bracket_g[low], sm.g_new);
    }
  }
  *t_io = br[low];
  copy(sm.g, sm.bracket_g[low]);
  *ls_evals = evals;
  return br_f[low];
}

struct Args {
  const double* total_sc;
  const double* snv_sc;
  const double* elbo_draws;        // [64][194]
  const double* mean_draws;        // [1000][194]
  double* rates_out;               // [n][12][16]
  double* mu_out;                  // [n][194] or null
  double* log_sigma_out;
  int32_t* n_iter_out;             // [n] or null
  int32_t* func_evals_out;
  unsigned char* history;          // [n][2][100][388] doubles
};

__global__ void __launch_bounds__(NT, 1) snv_context_fit_kernel(Args a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x;
  const size_t problem = blockIdx.x;
  const double* eps = a.elbo_draws;
  double* Y = reinterpret_cast<double*>(a.history + problem * HISTORY_BYTES);   // old_dirs
  double* Sv = Y + (size_t)HISTORY * P;                                          // old_stps
  for (int i = tid; i < CELLS; i += NT) {
    const double tot = a.total_sc[problem * CELLS + i], k = a.snv_sc[problem * CELLS + i];
    sm.total[i] = tot;
    sm.snv[i] = k < tot ? k : tot;                         // torch.minimum(snv, total)
  }
  __syncthreads();
  // the smoothed maximum-likelihood start; row sums of the integer counts are exact in any order
  double* row_snv = sm.row_g;
  if (tid < S) {
    double r = 0.0;
    for (int c = 0; c < CX; ++c) r += sm.snv[tid * CX + c];
    row_snv[tid] = r;
  }
  __syncthreads();
  if (tid < S) {
    const int s = tid;
    double lt[CX], mean = 0.0;
    for (int c = 0; c < CX; ++c) {
      lt[c] = log((sm.snv[s * CX + c] + 1.0) / (row_snv[s] + CX));
      mean += lt[c];
    }
    mean /= CX;
    for (int c = 0; c < CX - 1; ++c) sm.x[3 + (S - 1) + s * (CX - 1) + c] = lt[c] - mean;
  } else if (tid == 32) {
    double snv_sum = 0.0, tot_sum = 0.0;
    for (int i = 0; i < CELLS; ++i) {
      snv_sum += sm.snv[i];
      tot_sum += sm.total[i];
    }
    const double overall = (snv_sum + 1.0) / (tot_sum + 1e6);
    sm.x[0] = log(overall) - log1p(-overall);
    sm.x[1] = sm.x[2] = 0.0;
    double lt[S], mean = 0.0;
    for (int s = 0; s < S; ++s) {
      lt[s] = log((row_snv[s] + 1.0) / (snv_sum + S));
      mean += lt[s];
    }
    mean /= S;
    for (int s = 0; s < S - 1; ++s) sm.x[3 + s] = lt[s] - mean;
  }
  for (int j = D + tid; j < P; j += NT) sm.x[j] = -2.0;
  __syncthreads();

  // torch.optim.LBFGS.step
  double f = evaluate(sm, sm.x, sm.g, eps);
  int func_evals = 1, current_evals = 1, n_iter = 0;
  if (!(abs_max(sm.g, 1.0, sm.red) <= TOL_GRAD)) {
    int head = 0, num_old = 0;
    double H_diag = 1.0, t = 0.0;
    while (n_iter < MAX_ITER) {
      ++n_iter;
      if (n_iter == 1) {
        for (int j = tid; j < P; j += NT) sm.dir[j] = -sm.g[j];
      } else {
        double* y = sm.g_new;              // free between line searches
        double* s = sm.g_prev;
        for (int j = tid; j < P; j += NT) {
          y[j] = sm.g[j] - sm.prev_g[j];
          s[j] = sm.dir[j] * t;
        }
        const double ys = dot(y, s, sm.red);
        if (ys > 1e-10) {
          if (num_old == HISTORY) {
            head = (head + 1) % HISTORY;
            --num_old;
          }
          const int slot = (head + num_old) % HISTORY;
          for (int j = tid; j < P; j += NT) {
            Y[(size_t)slot * P + j] = y[j];
            Sv[(size_t)slot * P + j] = s[j];
          }
          if (tid == 0) sm.ro[slot] = 1.0 / ys;
          ++num_old;
          H_diag = ys / dot(y, y, sm.red);       // its barriers publish ro[slot]
        }
        for (int j = tid; j < P; j += NT) sm.dir[j] = -sm.g[j];
        for (int i = num_old - 1; i >= 0; --i) {
          const int idx = (head + i) % HISTORY;
          const double al = dot(Sv + (size_t)idx * P, sm.dir, sm.red) * sm.ro[idx];
          if (tid == 0) sm.al[i] = al;
          for (int j = tid; j < P; j += NT) sm.dir[j] += -al * Y[(size_t)idx * P + j];
        }
        for (int j = tid; j < P; j += NT) sm.dir[j] *= H_diag;
        for (int i = 0; i < num_old; ++i) {
          const int idx = (head + i) % HISTORY;
          const double be = dot(Y + (size_t)idx * P, sm.dir, sm.red) * sm.ro[idx];
          const double c = sm.al[i] - be;
          for (int j = tid; j < P; j += NT) sm.dir[j] += c * Sv[(size_t)idx * P + j];
        }
      }
      copy(sm.prev_g, sm.g);
      const double prev_loss = f;
      if (n_iter == 1) {
        double s = 0.0;
        for (int j = tid; j < P; j += NT) s += fabs(sm.g[j]);
        t = py_min(1.0, 1.0 / block_sum(s, sm.red));
      } else {
        t = 1.0;
      }
      const double gtd = dot(sm.g, sm.dir, sm.red);
      if (gtd > -TOL_CHANGE) break;
      int ls_evals = 0;
      f = strong_wolfe(sm, eps, &t, f, gtd, MAX_EVAL - current_evals, &ls_evals);
      for (int j = tid; j < P; j += NT) sm.x[j] = step_to(sm.x[j], t, sm.dir[j]);
      const bool opt_cond = abs_max(sm.g, 1.0, sm.red) <= TOL_GRAD;
      current_evals += ls_evals;
      func_evals += ls_evals;
      if (n_iter == MAX_ITER) break;
      if (current_evals >= MAX_EVAL) break;
      if (opt_cond) break;
      if (abs_max(sm.dir, t, sm.red) <= TOL_CHANGE) break;
      if (fabs(f - prev_loss) < TOL_CHANGE) break;
    }
  }
  __syncthreads();
  if (tid == 0) {
    if (a.n_iter_out) a.n_iter_out[problem] = n_iter;
    if (a.func_evals_out) a.func_evals_out[problem] = func_evals;
  }
  for (int j = tid; j < D; j += NT) {
    if (a.mu_out) a.mu_out[problem * D + j] = sm.x[j];
    if (a.log_sigma_out) a.log_sigma_out[problem * D + j] = sm.x[D + j];
    sm.sig[j] = exp(sm.x[D + j]);
  }
  // E_q[rate_sc]: the mean of exp(clamped log_rate) over the mean draws, 64 at a time, each cell summed in draw order
  double acc = 0.0;
  for (int first = 0; first < MEAN_DRAWS; first += ELBO_DRAWS) {
    const int n = min(ELBO_DRAWS, MEAN_DRAWS - first);
    __syncthreads();
    if (tid < n) draw_scalars(sm, sm.x, a.mean_draws + (size_t)(first + tid) * D, tid, false);
    __syncthreads();
    for (int u = tid; u < n * S; u += NT) {
      const int d = u / S, s = u % S;
      double lx[CX];
      context_simplex(sm, sm.x, a.mean_draws + (size_t)(first + d) * D, s, lx);
      const double base = sm.log_r[d] + log((double)(S * CX)) + sm.log_ts[d * S + s];
      for (int c = 0; c < CX; ++c) {
        const double l = base + lx[c];
        sm.gz[(size_t)d * CELLS + s * CX + c] = exp(l <= MAX_LOG_RATE ? l : MAX_LOG_RATE);
      }
    }
    __syncthreads();
    if (tid < CELLS)
      for (int d = 0; d < n; ++d) acc += sm.gz[(size_t)d * CELLS + tid];
  }
  if (tid < CELLS) a.rates_out[problem * CELLS + tid] = acc / MEAN_DRAWS;
}

}  // namespace ctxfit

extern "C" size_t pmt_snv_context_fit_workspace_size(int32_t n) {
  if (n < 1) return 0;
  return (size_t)n * ctxfit::HISTORY_BYTES + 256;        // the extra 256 bytes realign a caller's buffer
}

extern "C" int pmt_snv_context_fit_many(int32_t n, const double* total_sc, const double* snv_sc, const double* elbo_draws,
                                        const double* mean_draws, double* rates_out, double* mu_out, double* log_sigma_out,
                                        int32_t* n_iter_out, int32_t* func_evals_out, void* workspace, size_t workspace_bytes,
                                        void* stream) {
  const char* who = "pmt_snv_context_fit_many";
  PMT_CHECK(n >= 1, "%s: n %d < 1", who, n);
  PMT_CHECK(total_sc, "%s: null total_sc", who);
  PMT_CHECK(snv_sc, "%s: null snv_sc", who);
  PMT_CHECK(elbo_draws, "%s: null elbo_draws", who);
  PMT_CHECK(mean_draws, "%s: null mean_draws", who);
  PMT_CHECK(rates_out, "%s: null rates_out", who);
  PMT_CHECK(workspace, "%s: null workspace", who);
  const size_t need = pmt_snv_context_fit_workspace_size(n);
  PMT_CHECK(workspace_bytes >= need, "%s: workspace too small: %zu bytes, need %zu", who, workspace_bytes, need);
  const size_t smem = sizeof(ctxfit::Smem);
  PMT_CUDA(cudaFuncSetAttribute(ctxfit::snv_context_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ctxfit::Args a{total_sc, snv_sc, elbo_draws, mean_draws, rates_out, mu_out, log_sigma_out, n_iter_out, func_evals_out,
                 pmt_align_up(workspace, 256)};
  ctxfit::snv_context_fit_kernel<<<n, ctxfit::NT, smem, reinterpret_cast<cudaStream_t>(stream)>>>(a);
  const cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "%s launch failed: %s", who, cudaGetErrorString(e));
  return 0;
}
