// Backward kernels of the ArtifactModel hot path (sm_100a) and the backward half of the C-ABI.
//
// pmt_backward = autograd of artifact_model.py:239-297 w.r.t. the flat materialised weights:
//   reads_backward_kernel     per tile: forward recompute (activations to a per-CTA L2-resident scratch),
//                             then head -> rotation -> reducer -> gated blocks -> read embedding in reverse;
//                             weight gradients accumulate in a CTA-private flat buffer (no atomics, fixed order)
//   reads_backward_long_kernel  the same pieces for sets longer than a tile, walked in chunks
//   info_mlp_backward_kernel  info_embedding MLP, rows = variants
//   hap_cnn_backward_kernel   DNASequenceConvolution
//   reduce_partials_kernel    sum of the CTA-private buffers in CTA order (bitwise reproducible)
//   skip_fix_kernel           DenseSkipBlock.alpha gradients and the alpha scaling of its last layer
#include <cstdio>
#include <cstring>

// The per-row phases are written for NPART = NTHREADS / TILE threads per tile row.  Measured on B200 (65 536 variants,
// profiles/r1_tensor_core_kernels.md): 256 threads 30.4 ms, 384 threads 31.6 ms, 512 threads 32.5 ms (register cap 128,
// spills), so NTHREADS stays at 256: two threads per row.
#include "pmt_cnn.cuh"
#include "pmt_call.h"
#include "pmt_tile.cuh"

namespace pmt {

struct BwdArgs {
  const float* wflat;
  const float* image;
  PmtBatch batch;
  const float* info_seq;      // [B][d_info + d_seq] from the variant kernels (forward recompute)
  const float* d_logits_bk;   // upstream gradients (may be null)
  const float* d_alt_means;
  const float* d_ref_means;
  float* d_info_seq;          // [B][d_info + d_seq] gradient handed to the variant kernels
  float* scratch;             // per-CTA activation scratch
  long long scratch_stride;   // floats
  float* long_scratch;        // per-CTA scratch of the long-set kernel (one region per chunk of the longest set)
  long long long_scratch_stride;
  float* partials;            // per-CTA flat gradient buffers [grid][n_params]
  int n_claims;
};

// The four activation buffers of a backward CTA, as (base, stride): an array of pointers would live in local memory,
// and with nearly all of L1 carved out as shared memory every read of it is an L2 round trip.
struct BufSet {
  float* base;
  int stride;   // floats
  __device__ __forceinline__ float* operator[](int i) const { return base + i * stride; }
};
__device__ __forceinline__ float* pick_free(const BufSet& bufs, const float* a, const float* b, const float* c) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float* p = bufs[i];
    if (p != a && p != b && p != c) return p;
  }
  return nullptr;
}

// Backward of an MLP program (mlp.py:8-76).  On entry `g` holds dL/d(output); activations entering each op
// were saved at scr + scr_off[i].  Returns the buffer holding dL/d(input) (meaningful if need_input_grad).
// Weight/bias gradients are accumulated into `part`; for the last layer of a DenseSkipBlock the un-scaled
// U = dx_out . s^T is accumulated instead (skip_fix_kernel turns it into dW = alpha U and d alpha = <W, U> + <b, Ub>).
static __device__ __noinline__ float* mlp_backward(const Plan& P, const PmtLinearOp* ops, int n_ops, int g0,
                                                   const float* scr, const int* scr_off, float* g, const BufSet& bufs,
                                                   Stage& stage, const float* wflat, float* part, int rows_used,
                                                   bool need_input_grad) {
  float* gcur = g;
  int i = n_ops - 1;
  while (i >= 0) {
    if (ops[i].flags & PMT_OP_SKIP_END) {
      const int j1 = i;
      int j0 = i;
      while (!(ops[j0].flags & PMT_OP_SKIP_BEGIN)) --j0;
      float* gres = gcur;
      float* din = gres;
      const float alpha = __ldg(wflat + ops[j1].alpha_off);
      for (int j = j1; j >= j0; --j) {
        const PmtLinearOp& lop = ops[j];
        const GemmOp& gop = P.gemm[g0 + j];
        float* A = pick_free(bufs, gres, din, nullptr);
        __syncthreads();
        load_rows_async(A, lop.in_dim, scr + scr_off[j]);   // acquire() waits for every cp.async of the thread
        const float* imgT = stage.acquire(MAX_GEMM + g0 + j);
        if (j == j0) { selu_copy(A, A, lop.in_dim); __syncthreads(); }   // A = s0 = SELU(x)
        if (j > 0) stage.prefetch(MAX_GEMM + g0 + j - 1);
        wgrad_tile(smem_addr(din), lop.out_dim, smem_addr(A), lop.in_dim, part + lop.w_off, 0, rows_used);
        rowdot_tile(din, nullptr, lop.out_dim, part + lop.b_off, 0, rows_used);
        const float scale = (j == j1) ? alpha : 1.f;
        float* dnext = pick_free(bufs, gres, din, A);
        gemm_tile_T(din, gop, imgT, 0, dnext, EPI_DSELU, scale, A, rows_used);
        if (j == j0) {   // gres += dnext (the SELU(x) branch joins the identity branch)
          __syncthreads();
          for (int t = threadIdx.x; t < lop.in_dim * (TILE / 4); t += NTHREADS) {
            const int f = t / (TILE / 4), q = t % (TILE / 4);
            float4 a = *reinterpret_cast<float4*>(gres + f * LD + q * 4);
            const float4 b = *reinterpret_cast<const float4*>(dnext + f * LD + q * 4);
            a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
            *reinterpret_cast<float4*>(gres + f * LD + q * 4) = a;
          }
        } else {
          din = dnext;
        }
      }
      if (j0 > 0 && (ops[j0 - 1].flags & PMT_OP_POST_SELU)) {   // x itself is a SELU output of the previous layer
        float* A = pick_free(bufs, gres, nullptr, nullptr);
        __syncthreads();
        load_rows(A, ops[j0].in_dim, scr + scr_off[j0]);
        __syncthreads();
        mul_dselu(gres, A, ops[j0].in_dim);
      }
      gcur = gres;
      i = j0 - 1;
    } else {
      const PmtLinearOp& lop = ops[i];
      const GemmOp& gop = P.gemm[g0 + i];
      float* A = pick_free(bufs, gcur, nullptr, nullptr);
      __syncthreads();
      load_rows(A, lop.in_dim, scr + scr_off[i]);
      const bool want_dgrad = i > 0 || need_input_grad;
      const float* imgT = nullptr;
      if (want_dgrad) {
        imgT = stage.acquire(MAX_GEMM + g0 + i);
        if (i > 0) stage.prefetch(MAX_GEMM + g0 + i - 1);
      } else {
        __syncthreads();
      }
      wgrad_tile(smem_addr(gcur), lop.out_dim, smem_addr(A), lop.in_dim, part + lop.w_off, 0, rows_used);
      rowdot_tile(gcur, nullptr, lop.out_dim, part + lop.b_off, 0, rows_used);
      if (want_dgrad) {
        float* dnext = pick_free(bufs, gcur, A, nullptr);
        const bool dselu = i > 0 && (ops[i - 1].flags & PMT_OP_POST_SELU);
        gemm_tile_T(gcur, gop, imgT, 0, dnext, dselu ? EPI_DSELU : EPI_STORE, 1.f, A, rows_used);
        gcur = dnext;
      }
      i -= 1;
    }
  }
  __syncthreads();
  return gcur;
}

__device__ __forceinline__ float ldg_or_zero(const float* p, long long i) { return p ? __ldg(p + i) : 0.f; }

// ------------------------------------------------------------------------------------------------
// Per-tile pieces of the read-path backward, shared by the tile kernel (whole variants packed into one
// tile) and the long-set kernel (one variant walked in chunks of TILE rows).  The only cross-read coupling
// is the per-variant mean field of each gated block (gated_mlp.py:236-248), so a block's backward splits
// into: bwd_block_gate (everything up to the sums of d gate over the set), bwd_block_meanfield (once per
// set) and bwd_block_finish (the rest, which needs the mean-field gradient of the whole set).
// ------------------------------------------------------------------------------------------------
struct BwdTile {
  const Plan& P;
  const BwdArgs& A;
  TileCtx& C;
  Stage& stage;
  BlockAccum& acc;
  BufSet bufs;          // four [bwd_rows][LD] activation buffers
  float* dsums;         // [nv][2][sum_w] gradients of the mean fields (same layout as C.sums)
  float* wpart;         // BlockAccum storage [NWARPS][acc_cap]
  float* small;         // [64] scratch for tiny reductions
  float* part;          // this CTA's flat gradient buffer
  int acc_cap;
};

struct BwdSmem {
  BufSet bufs;
  float *st0, *st1, *dsums, *wpart, *small;
  int acc_cap;
};

static_assert(sizeof(Plan) % 16 == 0, "Plan is copied to shared memory in 16-byte units");
__device__ __forceinline__ const Plan* stage_plan_in_smem(const Plan& param, float* smem) {
  const int* src = reinterpret_cast<const int*>(&param);
  int* dst = reinterpret_cast<int*>(smem);
  for (int i = threadIdx.x; i < (int)(sizeof(Plan) / sizeof(int)); i += NTHREADS) dst[i] = src[i];
  __syncthreads();
  return reinterpret_cast<const Plan*>(smem);
}

__device__ __forceinline__ void carve_bwd_smem(const Plan& P, float* smem, TileCtx& C, BwdSmem& S) {
  const PmtModelDesc& D = P.d;
  const int R = P.bwd_rows;
  S.bufs.base = smem; S.bufs.stride = R * LD;
  S.st0 = smem + 4 * R * LD;
  S.st1 = S.st0 + P.stage_floats;
  C.X = S.bufs[0]; C.T1 = S.bufs[1]; C.T2 = S.bufs[2];
  C.sums = S.st1 + P.stage_floats;
  S.dsums = C.sums + TILE * 2 * P.sum_w;
  C.llsum = S.dsums + TILE * 2 * P.sum_w;
  const int n_head = D.d_feat + D.n_clusters * D.d_feat + 5 * D.n_clusters;
  S.acc_cap = n_head > 8 ? n_head : 8;
  S.wpart = C.llsum + TILE * 2 * 16;
  S.small = S.wpart + NWARPS * S.acc_cap;
  C.HC = reinterpret_cast<HeadConst*>(S.small + 64);
  C.M = reinterpret_cast<TileMeta*>((reinterpret_cast<uintptr_t>(C.HC + 1) + 15) & ~uintptr_t(15));
}

// Reducer -> rotation -> clustering head (recompute, activations to `scr`), then their backward
// (feature_clustering.py:82-135, euclidean_transformation.py:19-20, artifact_model.py:258-259).
// C.X holds the reducer's input.  Returns the buffer holding dL/d(output of the last gated block).
static __device__ __forceinline__ float* bwd_tail(BwdTile& T, float* scr) {
  const Plan& P = T.P;
  const BwdArgs& A = T.A;
  TileCtx& C = T.C;
  const PmtModelDesc& D = P.d;
  const TileMeta& M = *C.M;
  const float* W = C.W;
  float* part = T.part;
  BlockAccum& acc = T.acc;
  const int tid = threadIdx.x, row = tid & (TILE - 1), rp = tid / TILE;
  const int E = D.d_feat, K = D.n_clusters, rows_used = C.rows_used;
  const int my_var = M.rowvar[row];
  const bool is_alt = row >= M.ref_pad;
  const PmtOutputs no_out{};
  float *Yb, *Fb;
  tile_tail(P, C, T.stage, no_out, false, scr, Yb, Fb);
  float* Lb = pick_free(T.bufs, Yb, Fb, T.bufs[3]);   // the third forward buffer (held the log-likelihoods)
  float* Xtra = T.bufs[3];

  for (int i = tid; i < NWARPS * T.acc_cap; i += NTHREADS) T.wpart[i] = 0.f;
  __syncthreads();
  {
    const bool live = is_alt && my_var >= 0;
    const long long v = live ? (long long)M.v0 + my_var : 0;
    // row-part p writes its share of d f into Lb rows [p*E, (p+1)*E)
    float* dfp = Lb + rp * E * LD;
    for (int e = 0; e < E; ++e) dfp[e * LD + row] = 0.f;
    if (rp == 0) {
      const float g0 = live ? ldg_or_zero(A.d_logits_bk, v * (K + 2) + 0) : 0.f;
      const float g1 = live ? ldg_or_zero(A.d_logits_bk, v * (K + 2) + 1) : 0.f;
      for (int e = 0; e < E; ++e) {
        const float s = C.HC->sigma[e], f = Fb[e * LD + row];
        float contrib = 0.f;
        if (live) {
          dfp[e * LD + row] += -g0 * f / (s * s) - g1 * f / (4.f * s * s);
          contrib = g0 * (-1.f / s + f * f / (s * s * s)) + g1 * (-1.f / s + f * f / (4.f * s * s * s));
        }
        acc.add(e, contrib);
      }
    }
    for (int k = rp; k < K; k += NPART) {
      const float* u = W + D.unit_ke + k * E;
      const float gk = live ? ldg_or_zero(A.d_logits_bk, v * (K + 2) + 2 + k) : 0.f;
      const float tau = __ldg(W + D.tau_k + k), lam = __ldg(W + D.lambda_k + k), sg = __ldg(W + D.emg_sigma_k + k),
                  mu = __ldg(W + D.mu_k + k);
      float p = 0.f;
      for (int e = 0; e < E; ++e) p = fmaf(Fb[e * LD + row], __ldg(u + e), p);
      float o2 = 0.f, odu = 0.f;
      for (int e = 0; e < E; ++e) {
        const float o = Fb[e * LD + row] - p * __ldg(u + e);
        o2 = fmaf(o, o, o2); odu = fmaf(o, __ldg(u + e), odu);
      }
      const float zarg = (C.HC->shift[k] - p) / C.HC->sqrt2_sigma[k];
      const float dlp = dlogerfc(zarg);
      const float dpar_dp = -dlp / C.HC->sqrt2_sigma[k] - lam;
      const float c_orth = -1.f / C.HC->two_tau2[k];
      for (int e = 0; e < E; ++e) {
        const float f = Fb[e * LD + row], ue = __ldg(u + e), o = f - p * ue;
        if (live) dfp[e * LD + row] += gk * (c_orth * (2.f * o - 2.f * odu * ue) + dpar_dp * ue);
        acc.add(E + k * E + e, gk * (c_orth * (-2.f * f * odu - 2.f * p * o) + dpar_dp * f));
      }
      const int base = E + K * E;
      acc.add(base + 0 * K + k, gk * (-(E - 1) / tau + o2 / (tau * tau * tau)));                       // tau
      acc.add(base + 1 * K + k, gk * (dlp / C.HC->sqrt2_sigma[k] + lam));                              // mu
      acc.add(base + 2 * K + k, gk * (dlp * (1.41421356237f * lam - zarg / sg) + lam * lam * sg));    // emg sigma
      acc.add(base + 3 * K + k, gk * (1.f / lam + dlp * sg * 0.70710678118f + mu + lam * sg * sg - p));  // lambda
      // the log cluster weight is added once per variant, after the sum over its reads (feature_clustering.py:115-116)
      acc.add(base + 4 * K + k, (live && M.alt_head && row == M.alt_start[my_var]) ? gk : 0.f);
    }
  }
  __syncthreads();
  acc.flush(part + D.sigma_e, 0, E);
  acc.flush(part + D.unit_ke, E, K * E);
  {
    const int base = E + K * E;
    const int offs[5] = {D.tau_k, D.mu_k, D.emg_sigma_k, D.lambda_k, D.logw_k};
    for (int q = 0; q < 5; ++q) acc.flush(part + offs[q], base + q * K, K);
  }
  // d f = head part (all row-parts) + mean part; written in place over the final features
  {
    const int e_lo = part_lo(E, rp), e_hi = part_lo(E, rp + 1);
    for (int e = e_lo; e < e_hi; ++e) {
      float d = 0.f;
#pragma unroll
      for (int q = 0; q < NPART; ++q) d += Lb[(q * E + e) * LD + row];
      if (my_var >= 0) {
        const long long v = (long long)M.v0 + my_var;
        d += is_alt ? ldg_or_zero(A.d_alt_means, v * E + e) / (M.alt_total[my_var] + 1e-4f)
                    : ldg_or_zero(A.d_ref_means, v * E + e) / (M.ref_total[my_var] + 1e-4f);
      } else {
        d = 0.f;
      }
      Fb[e * LD + row] = d;
      Yb[e * LD + row] += __ldg(W + D.translation + e);   // y + t, the rotation's input
    }
  }
  __syncthreads();
  // rotation (euclidean_transformation.py:19-20): f = Q (y + t)
  wgrad_tile(smem_addr(Fb), E, smem_addr(Yb), E, part + D.rotation, 0, rows_used);
  {
    const int e_lo = part_lo(E, rp), e_hi = part_lo(E, rp + 1);
    for (int j = e_lo; j < e_hi; ++j) {
      float a = 0.f;
      for (int i = 0; i < E; ++i) a = fmaf(__ldg(W + D.rotation + i * E + j), Fb[i * LD + row], a);
      Xtra[j * LD + row] = a;
    }
  }
  __syncthreads();
  rowdot_tile(Xtra, nullptr, E, part + D.translation, 0, rows_used);
  float* G = mlp_backward(P, D.red_ops, D.n_red_ops, P.red_g0, scr, P.scr_red, Xtra, T.bufs, T.stage, W, part, rows_used, true);
  return G;
}

struct RowNorm { float mean, rstd, mean2, rstd2; };

// Reloads x (-> Ab) and z (-> Cz[0, 2H)) of gated block `blk` from the recompute scratch -- or, when `cz_state` is given,
// the [0, 6H) rows bwd_block_gate left in Cz -- and redoes the block's LayerNorm: Ab = xhat, Bn = LN(x).
static __device__ __forceinline__ RowNorm bwd_block_reload(BwdTile& T, int blk, const float* scr, const float* cz_state,
                                                           float* Ab, float* Bn, float* Cz, int prefetch_key) {
  const Plan& P = T.P;
  const PmtModelDesc& D = P.d;
  const PmtBlockOffsets& BO = D.blocks[blk];
  const float* W = T.C.W;
  const int row = threadIdx.x & (TILE - 1), rp = threadIdx.x / TILE;
  const int Dm = D.d_model, H = D.d_ffn / 2;
  load_rows_async(Ab, Dm, scr + P.scr_x[blk]);
  if (cz_state) load_rows_async(Cz, 6 * H, cz_state);
  else load_rows_async(Cz, 2 * H, scr + P.scr_z[blk]);
  cp_async_wait_all();
  T.stage.prefetch(prefetch_key);
  __syncthreads();
  RowNorm n;
  row_stats(Ab, Dm, row, n.mean, n.rstd);
  row_stats(Cz + H * LD, H, row, n.mean2, n.rstd2);
  __syncthreads();
  const int d_lo = part_lo(Dm, rp), d_hi = part_lo(Dm, rp + 1);
  for (int f = d_lo; f < d_hi; ++f) {
    const float xh = (Ab[f * LD + row] - n.mean) * n.rstd;
    Ab[f * LD + row] = xh;
    Bn[f * LD + row] = xh * __ldg(W + BO.ln_w + f) + __ldg(W + BO.ln_b + f);
  }
  return n;
}

// First half of a gated block's backward (gated_mlp.py:177-251 in reverse) over the rows of this tile: proj2, the
// gate, the scalar gate parameters, and the per-variant sums of d gate (into T.dsums; `accumulate` adds to them when
// the set spans several chunks).  `means`: the block's forward mean fields [2][sum_w] when the set spans several
// chunks (nullptr: computed here from the tile, which then holds whole sets).  Leaves Cz = [z1 z2 | xhat2 | gate | d z1 | d gate].
static __device__ __forceinline__ RowNorm bwd_block_gate(BwdTile& T, int blk, const float* scr, const float* means, float* G,
                                                         float* Ab, float* Bn, float* Cz, bool accumulate) {
  const Plan& P = T.P;
  TileCtx& C = T.C;
  const PmtModelDesc& D = P.d;
  const PmtBlockOffsets& BO = D.blocks[blk];
  const TileMeta& M = *C.M;
  const float* W = C.W;
  float* part = T.part;
  const int tid = threadIdx.x, row = tid & (TILE - 1), rp = tid / TILE;
  const int Dm = D.d_model, H = D.d_ffn / 2, rows_used = C.rows_used, ref_pad = M.ref_pad;
  const int my_var = M.rowvar[row];
  const bool is_alt = row >= ref_pad;
  const int g1 = P.blk_g0 + 2 * blk, g2 = g1 + 1;
  const float alpha = __ldg(W + (is_alt ? BO.alpha_alt : BO.alpha_ref));
  const float beta = __ldg(W + (is_alt ? BO.beta_alt : BO.beta_ref));
  const float gamma = __ldg(W + BO.gamma);
  const int f_lo = part_lo(H, rp), f_hi = part_lo(H, rp + 1);
  const RowNorm n = bwd_block_reload(T, blk, scr, nullptr, Ab, Bn, Cz, MAX_GEMM + g2);
  for (int f = f_lo; f < f_hi; ++f) {
    const float xh2 = (Cz[(H + f) * LD + row] - n.mean2) * n.rstd2;
    Cz[(2 * H + f) * LD + row] = xh2;
    Cz[(3 * H + f) * LD + row] = xh2 * __ldg(W + BO.ln2_w + f) + __ldg(W + BO.ln2_b + f);   // z2n
  }
  __syncthreads();
  if (means) {
    for (int i = tid; i < 2 * P.sum_w; i += NTHREADS) C.sums[i] = means[i];
    __syncthreads();
  } else {
    segment_sums(M, Cz, 3 * H, H, C.sums, P.sum_w, false, false);
    __syncthreads();
    block_means(P, C, blk);
  }
  for (int f = f_lo; f < f_hi; ++f) {
    const float gate = gate_value(P, C, BO, row, f, Cz[(3 * H + f) * LD + row], my_var, is_alt, alpha, beta, gamma);
    Cz[(3 * H + f) * LD + row] = gate;
    Cz[(4 * H + f) * LD + row] = Cz[f * LD + row] * gate;   // u = z1 * gate
  }
  // proj2: x_out = x + W2_s u + b2_s
  const float* imgT2 = T.stage.acquire(MAX_GEMM + g2);
  T.stage.prefetch(MAX_GEMM + g1);
  wgrad_tile(smem_addr(G), Dm, smem_addr(Cz + 4 * H * LD), H, part + BO.p2_ref_w, 0, ref_pad);
  wgrad_tile(smem_addr(G), Dm, smem_addr(Cz + 4 * H * LD), H, part + BO.p2_alt_w, ref_pad, rows_used);
  rowdot_tile(G, nullptr, Dm, part + BO.p2_ref_b, 0, ref_pad);
  rowdot_tile(G, nullptr, Dm, part + BO.p2_alt_b, ref_pad, rows_used);
  gemm_tile_T(G, P.gemm[g2], imgT2, ref_pad, Cz + 5 * H * LD, EPI_STORE, 1.f, nullptr, rows_used);   // du
  __syncthreads();
  {  // d z1 = du * gate ; d gate = du * z1 ; scalar gradients of the gate
    float s_alpha = 0.f, s_beta = 0.f, s_gamma = 0.f;
    for (int f = f_lo; f < f_hi; ++f) {
      const float du = Cz[(5 * H + f) * LD + row], gate = Cz[(3 * H + f) * LD + row], z1 = Cz[f * LD + row];
      const float dgate = du * z1;
      Cz[(4 * H + f) * LD + row] = du * gate;
      Cz[(5 * H + f) * LD + row] = dgate;
      if (my_var >= 0) {
        const float z2n = Cz[(2 * H + f) * LD + row] * __ldg(W + BO.ln2_w + f) + __ldg(W + BO.ln2_b + f);
        const float m_ref = C.sums[(my_var * 2 + 0) * P.sum_w + f];
        s_alpha = fmaf(dgate, z2n, s_alpha);
        s_beta = fmaf(dgate, is_alt ? C.sums[(my_var * 2 + 1) * P.sum_w + f] : m_ref, s_beta);
        if (is_alt) s_gamma = fmaf(dgate, m_ref, s_gamma);
      }
    }
    T.acc.add(0, is_alt ? 0.f : s_alpha); T.acc.add(1, is_alt ? s_alpha : 0.f);
    T.acc.add(2, is_alt ? 0.f : s_beta);  T.acc.add(3, is_alt ? s_beta : 0.f);
    T.acc.add(4, s_gamma);
  }
  __syncthreads();
  if (tid < 5) {
    const int off = tid == 0 ? BO.alpha_ref : (tid == 1 ? BO.alpha_alt : (tid == 2 ? BO.beta_ref : (tid == 3 ? BO.beta_alt : BO.gamma)));
    float s = 0.f;
    for (int w = 0; w < NWARPS; ++w) s += T.wpart[w * T.acc_cap + tid];
    red_add(part + off, s);
  }
  segment_sums(M, Cz, 5 * H, H, T.dsums, P.sum_w, false, accumulate);
  __syncthreads();
  return n;
}

// Gradients of the mean fields of block `blk` (ragged_sets.py:144-155 backward), once per set: T.dsums goes from the
// per-variant sums of d gate to d z2n's per-read share; C.sums holds the block's forward mean fields.
static __device__ __forceinline__ void bwd_block_meanfield(BwdTile& T, int blk) {
  const Plan& P = T.P;
  TileCtx& C = T.C;
  const PmtBlockOffsets& BO = P.d.blocks[blk];
  const TileMeta& M = *C.M;
  const float* W = C.W;
  float* dsums = T.dsums;
  const int tid = threadIdx.x, H = P.d.d_ffn / 2;
  const float gamma = __ldg(W + BO.gamma);
  const float regw = __ldg(W + BO.reg_weight) + 0.25f;
  const float b_ref = __ldg(W + BO.beta_ref), b_alt = __ldg(W + BO.beta_alt);
  for (int idx = tid; idx < M.nv * H; idx += NTHREADS) {
    const int j = idx / H, f = idx % H;
    const float s_ref = dsums[(j * 2 + 0) * P.sum_w + f], s_alt = dsums[(j * 2 + 1) * P.sum_w + f];
    dsums[(j * 2 + 0) * P.sum_w + f] = b_ref * s_ref + gamma * s_alt;   // d m_ref
    dsums[(j * 2 + 1) * P.sum_w + f] = b_alt * s_alt;                   // d m_alt
  }
  __syncthreads();
  if (tid < H) {
    float d_reg = 0.f, d_w = 0.f;
    const float reg = __ldg(W + BO.regularizer + tid);
    for (int j = 0; j < M.nv; ++j) {
      const float dm = dsums[(j * 2 + 0) * P.sum_w + tid], den = M.ref_total[j] + regw;
      d_reg += dm * regw / den;
      d_w += dm * (reg - C.sums[(j * 2 + 0) * P.sum_w + tid]) / den;
    }
    red_add(T.part + BO.regularizer + tid, d_reg);
    T.small[tid] = d_w;
  }
  __syncthreads();
  if (tid == 0) {
    float s = 0.f;
    for (int f = 0; f < H; ++f) s += T.small[f];
    red_add(T.part + BO.reg_weight, s);
  }
  for (int idx = tid; idx < M.nv * H; idx += NTHREADS) {
    const int j = idx / H, f = idx % H;
    dsums[(j * 2 + 0) * P.sum_w + f] /= (M.ref_total[j] + regw);
    dsums[(j * 2 + 1) * P.sum_w + f] /= (M.alt_total[j] + 1e-4f);
  }
  __syncthreads();
}

// Second half of a gated block's backward: SGU LayerNorm, proj1, the block's LayerNorm; G += dL/dx through the block.
// Expects Ab = xhat, Bn = LN(x), Cz as bwd_block_gate left it, and the row statistics of bwd_block_reload.
static __device__ __forceinline__ void bwd_block_finish(BwdTile& T, int blk, float* G, float* Ab, float* Bn, float* Cz,
                                                        const RowNorm& n) {
  const Plan& P = T.P;
  TileCtx& C = T.C;
  const PmtModelDesc& D = P.d;
  const PmtBlockOffsets& BO = D.blocks[blk];
  const TileMeta& M = *C.M;
  const float* W = C.W;
  float* part = T.part;
  float* dsums = T.dsums;
  const int row = threadIdx.x & (TILE - 1), rp = threadIdx.x / TILE;
  const int Dm = D.d_model, H = D.d_ffn / 2, rows_used = C.rows_used, ref_pad = M.ref_pad;
  const int my_var = M.rowvar[row];
  const bool is_alt = row >= ref_pad;
  const int g1 = P.blk_g0 + 2 * blk;
  const float alpha = __ldg(W + (is_alt ? BO.alpha_alt : BO.alpha_ref));
  const int f_lo = part_lo(H, rp), f_hi = part_lo(H, rp + 1);
  const int d_lo = part_lo(Dm, rp), d_hi = part_lo(Dm, rp + 1);
  for (int f = f_lo; f < f_hi; ++f) {   // d z2n
    float d = alpha * Cz[(5 * H + f) * LD + row];
    if (my_var >= 0) d += dsums[(my_var * 2 + (is_alt ? 1 : 0)) * P.sum_w + f];
    Cz[(3 * H + f) * LD + row] = d;
  }
  __syncthreads();
  rowdot_tile(Cz + 3 * H * LD, Cz + 2 * H * LD, H, part + BO.ln2_w, 0, rows_used);
  rowdot_tile(Cz + 3 * H * LD, nullptr, H, part + BO.ln2_b, 0, rows_used);
  {  // SGU LayerNorm backward -> d z2 (pre-norm), placed after d z1 so that [4H, 6H) = d z
    float m1 = 0.f, m2 = 0.f;
    for (int f = 0; f < H; ++f) {
      const float dxh = Cz[(3 * H + f) * LD + row] * __ldg(W + BO.ln2_w + f);
      m1 += dxh; m2 = fmaf(dxh, Cz[(2 * H + f) * LD + row], m2);
    }
    m1 /= H; m2 /= H;
    for (int f = f_lo; f < f_hi; ++f) {
      const float dxh = Cz[(3 * H + f) * LD + row] * __ldg(W + BO.ln2_w + f);
      Cz[(5 * H + f) * LD + row] = n.rstd2 * (dxh - m1 - Cz[(2 * H + f) * LD + row] * m2);
    }
  }
  __syncthreads();
  mul_dselu(Cz + 4 * H * LD, Cz, 2 * H);   // through z = SELU(proj1 n)
  // proj1: z_pre = W1_s n + b1_s
  const float* imgT1 = T.stage.acquire(MAX_GEMM + g1);
  if (blk > 0) T.stage.prefetch(MAX_GEMM + g1 - 1);
  wgrad_tile(smem_addr(Cz + 4 * H * LD), 2 * H, smem_addr(Bn), Dm, part + BO.p1_ref_w, 0, ref_pad);
  wgrad_tile(smem_addr(Cz + 4 * H * LD), 2 * H, smem_addr(Bn), Dm, part + BO.p1_alt_w, ref_pad, rows_used);
  rowdot_tile(Cz + 4 * H * LD, nullptr, 2 * H, part + BO.p1_ref_b, 0, ref_pad);
  rowdot_tile(Cz + 4 * H * LD, nullptr, 2 * H, part + BO.p1_alt_b, ref_pad, rows_used);
  __syncthreads();
  gemm_tile_T(Cz + 4 * H * LD, P.gemm[g1], imgT1, ref_pad, Bn, EPI_STORE, 1.f, nullptr, rows_used);   // d n
  __syncthreads();
  rowdot_tile(Bn, Ab, Dm, part + BO.ln_w, 0, rows_used);
  rowdot_tile(Bn, nullptr, Dm, part + BO.ln_b, 0, rows_used);
  {  // LayerNorm backward, added to the residual gradient
    float m1 = 0.f, m2 = 0.f;
    for (int f = 0; f < Dm; ++f) {
      const float dxh = Bn[f * LD + row] * __ldg(W + BO.ln_w + f);
      m1 += dxh; m2 = fmaf(dxh, Ab[f * LD + row], m2);
    }
    m1 /= Dm; m2 /= Dm;
    for (int f = d_lo; f < d_hi; ++f) {
      const float dxh = Bn[f * LD + row] * __ldg(W + BO.ln_w + f);
      G[f * LD + row] += n.rstd * (dxh - m1 - Ab[f * LD + row] * m2);
    }
  }
  __syncthreads();
}

// concat (artifact_model.py:246-251): d info_seq of each variant (added to it when the set spans several chunks), then
// the read embedding's backward (artifact_model.py:243).  G = dL/d(input of the first gated block).
static __device__ __forceinline__ void bwd_embed(BwdTile& T, float* scr, float* G, bool accumulate) {
  const Plan& P = T.P;
  const PmtModelDesc& D = P.d;
  const TileMeta& M = *T.C.M;
  {
    const int w = D.d_info + D.d_seq;
    for (int idx = threadIdx.x; idx < M.nv * w; idx += NTHREADS) {
      const int j = idx / w, f = idx % w;
      const float* p = G + (D.d_read + f) * LD;
      float s = 0.f;
      for (int i = 0; i < M.ref_cnt[j]; ++i) s += p[M.ref_start[j] + i];
      for (int i = 0; i < M.alt_cnt[j]; ++i) s += p[M.alt_start[j] + i];
      float* o = T.A.d_info_seq + ((long long)M.v0 + j) * w + f;
      *o = accumulate ? *o + s : s;
    }
  }
  mlp_backward(P, D.read_ops, D.n_read_ops, P.read_g0, scr, P.scr_read, G, T.bufs, T.stage, T.C.W, T.part, T.C.rows_used, false);
  __syncthreads();
}

__global__ void __launch_bounds__(NTHREADS, 1)
reads_backward_kernel(const __grid_constant__ Plan Pparam, const __grid_constant__ BwdArgs A) {
  extern __shared__ __align__(16) float smem_all[];
  // The plan is indexed dynamically everywhere (layer tables, GEMM descriptors, scratch offsets); from the kernel's
  // parameter bank every such read is a constant-cache round trip (1-2.5 k cycles per GEMM call went to them), so it
  // lives in shared memory.
  const Plan& P = *stage_plan_in_smem(Pparam, smem_all);
  float* smem = smem_all + sizeof(Plan) / sizeof(float);
  const PmtModelDesc& D = P.d;
  TileCtx C;
  BwdSmem S;
  carve_bwd_smem(P, smem, C, S);
  TileMeta& M = *C.M;
  C.W = A.wflat;
  BlockAccum acc;
  acc.init(S.wpart, S.acc_cap);
  const int tid = threadIdx.x;
  const int B = A.batch.n_variants, Dm = D.d_model, H = D.d_ffn / 2;
  Stage stage;
  stage.init(S.st0, S.st1, A.image, &P);
  if (tid == 0) head_constants(D, C.W, C.HC);
  for (int i = tid; i < 4 * P.bwd_rows * LD; i += NTHREADS) smem[i] = 0.f;
  __syncthreads();
  const long long total_ref = __ldg(A.batch.ref_off + B);
  float* scr = A.scratch + (long long)blockIdx.x * A.scratch_stride;
  BwdTile T{P, A, C, stage, acc, S.bufs, S.dsums, S.wpart, S.small, A.partials + (long long)blockIdx.x * D.n_params, S.acc_cap};
  const int claim = P.claim_variants;

  // static round-robin assignment of claims to CTAs: the summation order of every gradient is fixed
  for (int c = blockIdx.x; c < A.n_claims; c += gridDim.x) {
    const long long cv0 = (long long)c * claim;
    const int cv1 = (int)min((long long)B, cv0 + claim);
    int v_cur = (int)cv0;
    while (v_cur < cv1) {
      const int nv = build_tile(A.batch, v_cur, cv1, total_ref, M);
      if (nv == 0) { v_cur += 1; continue; }   // a set longer than a tile: reads_backward_long_kernel
      v_cur += nv;
      C.rows_used = (M.rows + 3) & ~3;

      // ======================= forward recompute, activations to scratch =======================
      tile_embed(P, C, stage, A.batch, A.info_seq, scr);
      for (int blk = 0; blk < D.n_blocks; ++blk) {
        save_rows(C.X, Dm, scr + P.scr_x[blk]);
        block_phase_a(P, C, stage, blk, scr + P.scr_z[blk]);
        segment_sums(M, C.T2, H, H, C.sums, P.sum_w, false, false);
        __syncthreads();
        block_means(P, C, blk);
        block_phase_b(P, C, stage, blk, blk + 1 < D.n_blocks ? P.blk_g0 + 2 * blk + 2 : P.red_g0);
      }
      // ======================= backward =======================
      float* G = bwd_tail(T, scr);
      float* const Ab = pick_free(S.bufs, G, nullptr, nullptr);
      float* const Bn = pick_free(S.bufs, G, Ab, nullptr);
      float* const Cz = pick_free(S.bufs, G, Ab, Bn);
      for (int blk = D.n_blocks - 1; blk >= 0; --blk) {
        const RowNorm n = bwd_block_gate(T, blk, scr, nullptr, G, Ab, Bn, Cz, false);
        bwd_block_meanfield(T, blk);
        bwd_block_finish(T, blk, G, Ab, Bn, Cz, n);
      }
      bwd_embed(T, scr, G, false);
    }
  }
}

// Sets longer than a tile (synthetic high-depth data, BASELINE config 5; real data is capped at 10 + 15 reads at ingest).
// One CTA walks a variant in chunks of TILE rows, every chunk with its own recompute scratch (plus the running dL/dx
// and the gate state of the block being differentiated); the mean fields and their gradients are accumulated over
// the chunks between the two halves of each block's backward, exactly where reads_forward_long_kernel accumulates them.
__global__ void __launch_bounds__(NTHREADS, 1)
reads_backward_long_kernel(const __grid_constant__ Plan Pparam, const __grid_constant__ BwdArgs A) {
  extern __shared__ __align__(16) float smem_all[];
  // The plan is indexed dynamically everywhere (layer tables, GEMM descriptors, scratch offsets); from the kernel's
  // parameter bank every such read is a constant-cache round trip (1-2.5 k cycles per GEMM call went to them), so it
  // lives in shared memory.
  const Plan& P = *stage_plan_in_smem(Pparam, smem_all);
  float* smem = smem_all + sizeof(Plan) / sizeof(float);
  const PmtModelDesc& D = P.d;
  TileCtx C;
  BwdSmem S;
  carve_bwd_smem(P, smem, C, S);
  TileMeta& M = *C.M;
  C.W = A.wflat;
  BlockAccum acc;
  acc.init(S.wpart, S.acc_cap);
  const int tid = threadIdx.x;
  const int B = A.batch.n_variants, Dm = D.d_model, H = D.d_ffn / 2;
  Stage stage;
  stage.init(S.st0, S.st1, A.image, &P);
  if (tid == 0) head_constants(D, C.W, C.HC);
  for (int i = tid; i < 4 * P.bwd_rows * LD; i += NTHREADS) smem[i] = 0.f;
  __syncthreads();
  const long long total_ref = __ldg(A.batch.ref_off + B);
  float* scr0 = A.long_scratch + (long long)blockIdx.x * A.long_scratch_stride;
  BwdTile T{P, A, C, stage, acc, S.bufs, S.dsums, S.wpart, S.small, A.partials + (long long)blockIdx.x * D.n_params, S.acc_cap};
  // per-chunk scratch: the recompute images of the tile kernel, then dL/dx [Dm] and the gate state [6H]
  const long long g_off = P.scratch_floats, cz_off = g_off + (long long)Dm * LD, chunk_stride = cz_off + 6LL * H * LD;
  float* const G = S.bufs[0];
  float* const Ab = S.bufs[1];
  float* const Bn = S.bufs[2];
  float* const Cz = S.bufs[3];
  const int sw2 = 2 * P.sum_w;

  for (int v = blockIdx.x; v < B; v += gridDim.x) {   // static assignment: fixed summation order
    const long long nref = __ldg(A.batch.ref_off + v + 1) - __ldg(A.batch.ref_off + v);
    const long long nalt = __ldg(A.batch.alt_off + v + 1) - __ldg(A.batch.alt_off + v);
    const long long total = ((nref + 3) & ~3LL) + nalt;
    if (total <= TILE) continue;
    const int n_chunks = (int)((total + TILE - 1) / TILE);
#define PMT_CHUNK(c)                                   \
    build_chunk(A.batch, v, (c), total_ref, M);        \
    C.rows_used = (M.rows + 3) & ~3;                   \
    float* scr = scr0 + (long long)(c) * chunk_stride;

    // ======================= forward recompute =======================
    for (int c = 0; c < n_chunks; ++c) {
      PMT_CHUNK(c)
      tile_embed(P, C, stage, A.batch, A.info_seq, scr);
      save_rows(C.X, Dm, scr + P.scr_x[0]);
      __syncthreads();
    }
    for (int blk = 0; blk < D.n_blocks; ++blk) {
      for (int c = 0; c < n_chunks; ++c) {
        PMT_CHUNK(c)
        load_rows(C.X, Dm, scr + P.scr_x[blk]);
        __syncthreads();
        block_phase_a(P, C, stage, blk, scr + P.scr_z[blk]);
        segment_sums(M, C.T2, H, H, C.sums, P.sum_w, false, c > 0);
        __syncthreads();
      }
      block_means(P, C, blk);
      for (int i = tid; i < sw2; i += NTHREADS) C.sums[(1 + blk) * sw2 + i] = C.sums[i];   // kept for the backward
      __syncthreads();
      for (int c = 0; c < n_chunks; ++c) {
        PMT_CHUNK(c)
        load_rows(C.X, Dm, scr + P.scr_x[blk]);
        load_rows(C.T2, 2 * H, scr + P.scr_z[blk]);
        __syncthreads();
        sgu_layernorm(P, C, blk);
        block_phase_b(P, C, stage, blk, -1);
        save_rows(C.X, Dm, blk + 1 < D.n_blocks ? scr + P.scr_x[blk + 1] : scr + P.scr_red[0]);
        __syncthreads();
      }
    }
    // ======================= backward =======================
    for (int c = 0; c < n_chunks; ++c) {
      PMT_CHUNK(c)
      load_rows(C.X, Dm, scr + P.scr_red[0]);
      __syncthreads();
      float* g = bwd_tail(T, scr);
      save_rows(g, Dm, scr + g_off);
      __syncthreads();
    }
    for (int blk = D.n_blocks - 1; blk >= 0; --blk) {
      for (int c = 0; c < n_chunks; ++c) {
        PMT_CHUNK(c)
        load_rows(G, Dm, scr + g_off);
        bwd_block_gate(T, blk, scr, C.sums + (1 + blk) * sw2, G, Ab, Bn, Cz, c > 0);
        save_rows(Cz, 6 * H, scr + cz_off);
        __syncthreads();
      }
      bwd_block_meanfield(T, blk);
      for (int c = 0; c < n_chunks; ++c) {
        PMT_CHUNK(c)
        load_rows(G, Dm, scr + g_off);
        const RowNorm n = bwd_block_reload(T, blk, scr, scr + cz_off, Ab, Bn, Cz, MAX_GEMM + P.blk_g0 + 2 * blk);
        bwd_block_finish(T, blk, G, Ab, Bn, Cz, n);
        save_rows(G, Dm, scr + g_off);
        __syncthreads();
      }
    }
    for (int c = 0; c < n_chunks; ++c) {
      PMT_CHUNK(c)
      load_rows(G, Dm, scr + g_off);
      __syncthreads();
      bwd_embed(T, scr, G, c > 0);
    }
#undef PMT_CHUNK
  }
}

// ------------------------------------------------------------------------------------------------
// info MLP backward: rows of the tile are variants
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NTHREADS, 1)
info_mlp_backward_kernel(const __grid_constant__ Plan P, const float* __restrict__ wflat, const float* __restrict__ image,
                         const void* __restrict__ info, int info_kind, long long info_stride, int n_variants,
                         const float* __restrict__ d_info_seq, float* scratch, long long scratch_stride, float* partials,
                         int rows_per_buf) {
  extern __shared__ __align__(16) float smem[];
  const BufSet bufs{smem, rows_per_buf * LD};
  float* st0 = smem + 4 * rows_per_buf * LD;
  float* st1 = st0 + P.info_stage_floats;
  Stage stage;
  stage.init(st0, st1, image, &P);
  float* scr = scratch + (long long)blockIdx.x * scratch_stride;
  float* part = partials + (long long)blockIdx.x * P.d.n_params;
  const int I = P.d.n_info_features, w = P.d.d_info + P.d.d_seq;
  for (int i = threadIdx.x; i < 4 * rows_per_buf * LD; i += NTHREADS) smem[i] = 0.f;
  __syncthreads();
  const int n_tiles = (n_variants + TILE - 1) / TILE;
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int v0 = t * TILE;
    const int nv = min(TILE, n_variants - v0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < TILE * I; idx += NTHREADS) {
      const int r = idx / I, f = idx % I;
      float v = 0.f;
      if (r < nv) {
        const long long off = (long long)(v0 + r) * info_stride + f;
        v = info_kind == PMT_F16 ? __half2float(reinterpret_cast<const __half*>(info)[off])
                                 : reinterpret_cast<const float*>(info)[off];
      }
      bufs[0][f * LD + r] = v;
    }
    float* out = run_mlp(P, P.d.info_ops, P.d.n_info_ops, P.info_g0, bufs[0], bufs[1], bufs[2], bufs[0], stage, wflat,
                         TILE, -1, scr, P.scr_info);
    __syncthreads();
    float* g = bufs[3];
    (void)out;
    for (int idx = threadIdx.x; idx < TILE * P.d.d_info; idx += NTHREADS) {
      const int r = idx / P.d.d_info, j = idx % P.d.d_info;
      g[j * LD + r] = r < nv ? d_info_seq[(long long)(v0 + r) * w + j] : 0.f;
    }
    __syncthreads();
    mlp_backward(P, P.d.info_ops, P.d.n_info_ops, P.info_g0, scr, P.scr_info, g, bufs, stage, wflat, part, TILE, false);
  }
}

// ------------------------------------------------------------------------------------------------
// reduction of the CTA-private gradient buffers, DenseSkipBlock fix-ups
// ------------------------------------------------------------------------------------------------
__global__ void reduce_partials_kernel(const float* __restrict__ partials, int n_cta, int n_params, float* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_params) return;
  float s = 0.f;
  for (int c = 0; c < n_cta; ++c) s += partials[(long long)c * n_params + p];
  out[p] = s;
}

// out holds U (un-scaled last-layer gradients of each DenseSkipBlock): d alpha = <W, U> + <b, Ub>; dW = alpha U.
__global__ void skip_fix_kernel(const __grid_constant__ Plan P, const float* __restrict__ w, float* __restrict__ out) {
  const SkipFix f = P.skipfix[blockIdx.x];
  __shared__ float red[256];
  float s = 0.f;
  for (int i = threadIdx.x; i < f.n_w; i += blockDim.x) s = fmaf(w[f.w_off + i], out[f.w_off + i], s);
  for (int i = threadIdx.x; i < f.n_b; i += blockDim.x) s = fmaf(w[f.b_off + i], out[f.b_off + i], s);
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  const float alpha = w[f.alpha_off];
  if (threadIdx.x == 0) out[f.alpha_off] = red[0];
  for (int i = threadIdx.x; i < f.n_w; i += blockDim.x) out[f.w_off + i] *= alpha;
  for (int i = threadIdx.x; i < f.n_b; i += blockDim.x) out[f.b_off + i] *= alpha;
}

// ------------------------------------------------------------------------------------------------
// haplotype CNN backward (dna_sequence_convolution.py:57-111).  VT variants per pass; every layer's
// activation of the pass stays in shared memory, channel-major with a per-variant stride lp[i] (multiple of 4)
// and a channel stride ld[i] == 4 (mod 32) so that 16-byte loads by lanes on consecutive channels are
// conflict-free (CnnBwdGeom, pmt_call.h).  conv data gradient = the forward conv routine on the zero-padded output
// gradient with the flipped/transposed image; conv weight gradient = register-tiled reduction over (variant, position).
// ------------------------------------------------------------------------------------------------

// Walks idx = tid, tid + NTHREADS, ... of a [C][V][L] index space keeping (c, v, p) without per-element integer
// divisions (they were a quarter of this kernel's instructions).
struct Idx3 {
  int c, v, p, sc, sv, sp, V, L;
  __device__ __forceinline__ Idx3(int V_, int L_) : V(V_), L(L_) {
    const int t = threadIdx.x;
    p = t % L_; v = (t / L_) % V_; c = t / (V_ * L_);
    sp = NTHREADS % L_; sv = (NTHREADS / L_) % V_; sc = NTHREADS / (V_ * L_);
  }
  __device__ __forceinline__ void next() {
    p += sp; v += sv; c += sc;
    if (p >= L) { p -= L; v += 1; }
    if (v >= V) { v -= V; c += 1; }
  }
};

__device__ __forceinline__ float act_grad_from_out(float y, int act) {
  if (act == PMT_ACT_SELU) return selu_grad_from_out(y);
  if (act == PMT_ACT_LEAKY_RELU) return y > 0.f ? 1.f : 0.01f;
  return 1.f;
}

__device__ __forceinline__ void stage_image(float* dst, const float* __restrict__ src, int n_floats) {
  for (int i = threadIdx.x; i < n_floats / 4; i += NTHREADS)
    reinterpret_cast<float4*>(dst)[i] = __ldg(reinterpret_cast<const float4*>(src) + i);
}

// dW[co][ci][t] += sum_{v, p} g[co][v, p] * in[ci][v, p + t];  g must be zero at padding positions.
// One (WG_OC output channels, 1 input channel) unit per thread; lanes run over consecutive input channels.
constexpr int WG_OC = NTHREADS >= 512 ? 2 : 4;
template <int KS>
__device__ __forceinline__ void conv_wgrad(const PmtCnnOp& op, const float* __restrict__ in, int in_ld, int lp_in,
                                           const float* __restrict__ g, int g_ld, int lp_out, int vt,
                                           float* __restrict__ part) {
  const int n_cg = (op.out_ch + WG_OC - 1) / WG_OC;
  for (int unit = threadIdx.x; unit < n_cg * op.in_ch; unit += NTHREADS) {
    const int cg = unit / op.in_ch, ci = unit % op.in_ch;
    float acc[WG_OC][KS];
#pragma unroll
    for (int b = 0; b < WG_OC; ++b)
#pragma unroll
      for (int t = 0; t < KS; ++t) acc[b][t] = 0.f;
    const float* xr = in + ci * in_ld;
    const float* gr[WG_OC];
#pragma unroll
    for (int b = 0; b < WG_OC; ++b) gr[b] = g + min(cg * WG_OC + b, op.out_ch - 1) * g_ld;
    for (int v = 0; v < vt; ++v) {
      for (int p0 = 0; p0 < lp_out; p0 += 4) {
        float xw[12];
        const float4 a = *reinterpret_cast<const float4*>(xr + v * lp_in + p0);
        xw[0] = a.x; xw[1] = a.y; xw[2] = a.z; xw[3] = a.w;
        if (KS > 1) {
          const float4 c = *reinterpret_cast<const float4*>(xr + v * lp_in + p0 + 4);
          xw[4] = c.x; xw[5] = c.y; xw[6] = c.z; xw[7] = c.w;
        }
        if (KS > 5) {
          const float4 c = *reinterpret_cast<const float4*>(xr + v * lp_in + p0 + 8);
          xw[8] = c.x; xw[9] = c.y; xw[10] = c.z; xw[11] = c.w;
        }
#pragma unroll
        for (int b = 0; b < WG_OC; ++b) {
          const float4 gv = *reinterpret_cast<const float4*>(gr[b] + v * lp_out + p0);
#pragma unroll
          for (int t = 0; t < KS; ++t) {
            acc[b][t] = fmaf(gv.x, xw[t], acc[b][t]);
            acc[b][t] = fmaf(gv.y, xw[t + 1], acc[b][t]);
            acc[b][t] = fmaf(gv.z, xw[t + 2], acc[b][t]);
            acc[b][t] = fmaf(gv.w, xw[t + 3], acc[b][t]);
          }
        }
      }
    }
#pragma unroll
    for (int b = 0; b < WG_OC; ++b) {
      const int co = cg * WG_OC + b;
      if (co < op.out_ch) {
#pragma unroll
        for (int t = 0; t < KS; ++t) red_add(part + op.w_off + (co * op.in_ch + ci) * KS + t, acc[b][t]);
      }
    }
  }
}

__global__ void __launch_bounds__(NTHREADS, 1)
hap_cnn_backward_kernel(const __grid_constant__ Plan P, const __grid_constant__ CnnGeom Gm_param,
                        const __grid_constant__ CnnBwdGeom Gb_param, const float* __restrict__ wflat,
                        const float* __restrict__ conv_image, const void* __restrict__ haps, int hap_kind,
                        long long hap_stride, int n_variants, const float* __restrict__ d_info_seq, float* partials) {
  extern __shared__ __align__(16) float smem[];
  // layer tables and geometry are indexed by the layer loop: from the parameter bank each read is a constant-cache
  // round trip (14 % of this kernel's stall samples sat on the two layer loops), so they are copied to shared memory
  __shared__ PmtCnnOp s_ops[PMT_MAX_CNN_OPS];
  __shared__ CnnBwdGeom s_gb;
  __shared__ CnnGeom s_gm;
  {
    const int* src_ops = reinterpret_cast<const int*>(P.d.cnn_ops);
    const int* src_gb = reinterpret_cast<const int*>(&Gb_param);
    const int* src_gm = reinterpret_cast<const int*>(&Gm_param);
    for (int i = threadIdx.x; i < (int)(sizeof(s_ops) / sizeof(int)); i += NTHREADS) reinterpret_cast<int*>(s_ops)[i] = src_ops[i];
    for (int i = threadIdx.x; i < (int)(sizeof(CnnBwdGeom) / sizeof(int)); i += NTHREADS) reinterpret_cast<int*>(&s_gb)[i] = src_gb[i];
    for (int i = threadIdx.x; i < (int)(sizeof(CnnGeom) / sizeof(int)); i += NTHREADS) reinterpret_cast<int*>(&s_gm)[i] = src_gm[i];
    __syncthreads();
  }
  const CnnBwdGeom& Gb = s_gb;
  const CnnGeom& Gm = s_gm;
  float* acts = smem;
  float* gA = acts + Gb.act_total;
  float* gB = gA + Gb.gbuf_floats;
  float* wst = gB + Gb.gbuf_floats;                        // staged conv image (forward or flipped)
  float* vec = wst + Gb.stage_floats;                      // [(n_linear + 1)][VT][vs] activations of the linear stack
  float* dvec = vec + (Gb.n_linear + 1) * Gb.vt * Gb.vs;   // [2][VT][vs] gradients of the linear stack
  const PmtModelDesc& D = P.d;
  const int VT = Gb.vt, VS = Gb.vs, L = D.hap_len, ns = Gb.n_spatial, tid = threadIdx.x;
  const int out_w = D.d_info + D.d_seq;
  float* part = partials + (long long)blockIdx.x * D.n_params;
  for (int i = tid; i < Gb.act_total + 2 * Gb.gbuf_floats; i += NTHREADS) smem[i] = 0.f;

  for (int v0 = blockIdx.x * VT; v0 < n_variants; v0 += gridDim.x * VT) {
    const int nv = min(VT, n_variants - v0);
    __syncthreads();
    // ---- forward recompute ----
    for (int idx = tid; idx < VT * 2 * L; idx += NTHREADS) {
      const int v = idx / (2 * L), hp = idx % (2 * L);
      int code = -1;
      if (v < nv) {
        const long long off = (long long)(v0 + v) * hap_stride + hp;
        code = hap_kind == PMT_I64 ? (int)reinterpret_cast<const long long*>(haps)[off]
                                   : (int)reinterpret_cast<const short*>(haps)[off];
      }
      const int h = hp / L, p = hp % L;
#pragma unroll
      for (int c = 0; c < 5; ++c) acts[Gb.act_off[0] + (2 * c + h) * Gb.ld[0] + v * Gb.lp[0] + p] = (code == c) ? 1.f : 0.f;
    }
    __syncthreads();
    for (int i = 0; i < ns; ++i) {
      const PmtCnnOp& op = s_ops[i];
      const float* in = acts + Gb.act_off[i];
      float* out = acts + Gb.act_off[i + 1];
      if (op.kind == PMT_CNN_CONV) {
        stage_image(wst, conv_image + Gm.img_off[i], op.in_ch * op.ksize * ((op.out_ch + 7) / 8) * GROUP_STRIDE);
        __syncthreads();
        PMT_CONV_DISPATCH(op.ksize, op, in, Gb.ld[i], Gb.lp[i], out, Gb.ld[i + 1], Gb.lp[i + 1], wst, wflat, VT)
      } else {
        const int lo = Gb.len[i + 1];
        Idx3 it(VT, lo);
        for (int idx = tid; idx < op.in_ch * VT * lo; idx += NTHREADS, it.next()) {
          const int c = it.c, v = it.v, p = it.p;
          const float* xr = in + c * Gb.ld[i] + v * Gb.lp[i] + p * op.stride;
          float m = xr[0];
          for (int t = 1; t < op.ksize; ++t) m = fmaxf(m, xr[t]);
          out[c * Gb.ld[i + 1] + v * Gb.lp[i + 1] + p] = m;
        }
      }
      __syncthreads();
    }
    // linear stack forward; vec level 0 = flattened spatial output (channel-major flatten)
    {
      const int C = Gb.ch[ns], len = Gb.len[ns];
      for (int idx = tid; idx < VT * C * len; idx += NTHREADS) {
        const int v = idx / (C * len), k = idx % (C * len), c = k / len, p = k % len;
        vec[v * VS + k] = acts[Gb.act_off[ns] + c * Gb.ld[ns] + v * Gb.lp[ns] + p];
      }
      __syncthreads();
      for (int l = 0; l < Gb.n_linear; ++l) {
        const PmtCnnOp& op = s_ops[ns + l];
        const float* vin = vec + l * VT * VS;
        float* vout = vec + (l + 1) * VT * VS;
        for (int idx = tid; idx < VT * op.out_ch; idx += NTHREADS) {
          const int v = idx / op.out_ch, n = idx % op.out_ch;
          float a = __ldg(wflat + op.b_off + n);
          const float* wr = wflat + op.w_off + (long long)n * op.in_ch;
          for (int k = 0; k < op.in_ch; ++k) a = fmaf(__ldg(wr + k), vin[v * VS + k], a);
          vout[v * VS + n] = apply_act(a, op.act);
        }
        __syncthreads();
      }
    }
    // ---- backward: linear stack ----
    float* dcur = dvec;
    float* dnxt = dvec + VT * VS;
    for (int idx = tid; idx < VT * D.d_seq; idx += NTHREADS) {
      const int v = idx / D.d_seq, n = idx % D.d_seq;
      dcur[v * VS + n] = v < nv ? d_info_seq[(long long)(v0 + v) * out_w + D.d_info + n] : 0.f;
    }
    __syncthreads();
    for (int l = Gb.n_linear - 1; l >= 0; --l) {
      const PmtCnnOp& op = s_ops[ns + l];
      const float* vin = vec + l * VT * VS;
      const float* vout = vec + (l + 1) * VT * VS;
      for (int idx = tid; idx < VT * op.out_ch; idx += NTHREADS) {
        const int v = idx / op.out_ch, n = idx % op.out_ch;
        dcur[v * VS + n] *= act_grad_from_out(vout[v * VS + n], op.act);
      }
      __syncthreads();
      for (int idx = tid; idx < op.out_ch * op.in_ch; idx += NTHREADS) {
        const int n = idx / op.in_ch, k = idx % op.in_ch;
        float a = 0.f;
        for (int v = 0; v < nv; ++v) a = fmaf(dcur[v * VS + n], vin[v * VS + k], a);
        red_add(part + op.w_off + idx, a);
      }
      for (int n = tid; n < op.out_ch; n += NTHREADS) {
        float a = 0.f;
        for (int v = 0; v < nv; ++v) a += dcur[v * VS + n];
        red_add(part + op.b_off + n, a);
      }
      for (int idx = tid; idx < VT * op.in_ch; idx += NTHREADS) {
        const int v = idx / op.in_ch, k = idx % op.in_ch;
        float a = 0.f;
        for (int n = 0; n < op.out_ch; ++n) a = fmaf(__ldg(wflat + op.w_off + (long long)n * op.in_ch + k), dcur[v * VS + n], a);
        dnxt[v * VS + k] = a;
      }
      __syncthreads();
      float* t = dcur; dcur = dnxt; dnxt = t;
    }
    // un-flatten into the gradient of the last spatial activation (layout of act[ns])
    float* gcur = gA;
    float* gnxt = gB;
    {
      const int C = Gb.ch[ns], len = Gb.len[ns];
      Idx3 it(VT, len);
      for (int idx = tid; idx < C * VT * len; idx += NTHREADS, it.next()) {
        const int c = it.c, v = it.v, p = it.p;
        gcur[c * Gb.ld[ns] + v * Gb.lp[ns] + p] = dcur[v * VS + c * len + p];
      }
      __syncthreads();
    }
    // ---- backward: spatial ops in reverse ----
    for (int i = ns - 1; i >= 0; --i) {
      const PmtCnnOp& op = s_ops[i];
      const float* in = acts + Gb.act_off[i];
      const float* out = acts + Gb.act_off[i + 1];
      const int li = Gb.len[i], lo = Gb.len[i + 1];
      const int ld_i = Gb.ld[i], lp_i = Gb.lp[i], ld_o = Gb.ld[i + 1], lp_o = Gb.lp[i + 1];
      if (op.kind == PMT_CNN_POOL) {
        // gradient goes to the first maximum of each window (one thread per INPUT element: no atomics)
        const int stride_shift = op.stride == 1 ? 0 : (op.stride == 2 ? 1 : -1);
        Idx3 it(VT, li);
        for (int idx = tid; idx < op.in_ch * VT * li; idx += NTHREADS, it.next()) {
          const int c = it.c, v = it.v, q = it.p;
          float a = 0.f;
          // windows p with p*stride <= q <= p*stride + ksize - 1 (shifts for the usual strides 1 and 2)
          int p_lo = q - op.ksize + 1;
          p_lo = p_lo <= 0 ? 0 : (stride_shift >= 0 ? (p_lo + op.stride - 1) >> stride_shift : (p_lo + op.stride - 1) / op.stride);
          const int p_hi = min(lo - 1, stride_shift >= 0 ? q >> stride_shift : q / op.stride);
          for (int p = p_lo; p <= p_hi; ++p) {
            const float* xr = in + c * ld_i + v * lp_i + p * op.stride;
            int arg = 0;
            float m = xr[0];
            for (int t = 1; t < op.ksize; ++t) if (xr[t] > m) { m = xr[t]; arg = t; }
            if (p * op.stride + arg == q) a += gcur[c * ld_o + v * lp_o + p];
          }
          gnxt[c * ld_i + v * lp_i + q] = a;
        }
        __syncthreads();
        float* t = gcur; gcur = gnxt; gnxt = t;
      } else {
        // through the activation folded into this conv; padding positions are forced to zero
        Idx3 it(VT, lp_o);
        for (int idx = tid; idx < op.out_ch * VT * lp_o; idx += NTHREADS, it.next()) {
          const int c = it.c, v = it.v, p = it.p;
          const int o = c * ld_o + v * lp_o + p;
          gcur[o] = p < lo ? gcur[o] * act_grad_from_out(out[o], op.act) : 0.f;
        }
        __syncthreads();
        switch (op.ksize) {
          case 1: conv_wgrad<1>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
          case 2: conv_wgrad<2>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
          case 3: conv_wgrad<3>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
          case 4: conv_wgrad<4>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
          case 5: conv_wgrad<5>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
          case 6: conv_wgrad<6>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
          case 7: conv_wgrad<7>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
          case 8: conv_wgrad<8>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
          default: conv_wgrad<9>(op, in, ld_i, lp_i, gcur, ld_o, lp_o, VT, part); break;
        }
        for (int co = tid; co < op.out_ch; co += NTHREADS) {
          float a = 0.f;
          for (int v = 0; v < VT; ++v)
            for (int p = 0; p < lo; ++p) a += gcur[co * ld_o + v * lp_o + p];
          red_add(part + op.b_off + co, a);
        }
        if (i > 0) {
          // zero-padded copy of the output gradient, then the forward conv routine with the flipped image
          const int ldg = Gb.ldg[i], lpg = Gb.lpg[i], ks = op.ksize;
          stage_image(wst, conv_image + Gm.img_total + Gm.imgT_off[i], op.out_ch * ks * ((op.in_ch + 7) / 8) * GROUP_STRIDE);
          Idx3 it(VT, lpg);
          for (int idx = tid; idx < op.out_ch * VT * lpg; idx += NTHREADS, it.next()) {
            const int c = it.c, v = it.v, pp = it.p, p = pp - (ks - 1);
            gnxt[c * ldg + v * lpg + pp] = (p >= 0 && p < lo) ? gcur[c * ld_o + v * lp_o + p] : 0.f;
          }
          __syncthreads();
          PmtCnnOp tr = op;
          tr.in_ch = op.out_ch; tr.out_ch = op.in_ch; tr.b_off = -1; tr.act = PMT_ACT_NONE;
          PMT_CONV_DISPATCH(ks, tr, gnxt, ldg, lpg, gcur, ld_i, lp_i, wst, wflat, VT)
          __syncthreads();
        }
      }
    }
  }
}

}  // namespace pmt

// ================================================================================================
// host side
// ================================================================================================
using namespace pmt;

static int pad_ld(int n) {   // smallest ld >= n + 12 with ld == 4 (mod 32)
  int ld = n + 12;
  while ((ld & 31) != 4) ++ld;
  return ld;
}

// The largest pass of variants (at most 16) whose activations, gradients and weight stage fit in shared memory.
static bool cnn_bwd_simt_geom(const Plan& P, const CnnGeom& G, CnnBwdGeom* out, size_t* smem_out, const char** why) {
  CnnBwdGeom& Gb = *out;
  const PmtModelDesc& d = P.d;
  const int ns = G.n_spatial;
  if (d.n_cnn_ops - ns < 1 || d.n_cnn_ops - ns > 4) {
    *why = "haplotype CNN backward supports 1..4 linear layers after flatten";
    return false;
  }
  size_t smem = 0;
  int vt = 16;
  for (; vt >= 1; --vt) {
    memset(&Gb, 0, sizeof(Gb));
    Gb.vt = vt; Gb.n_spatial = ns; Gb.n_linear = d.n_cnn_ops - ns;
    Gb.ch[0] = 10; Gb.len[0] = d.hap_len;
    for (int i = 0; i < ns; ++i) {
      const PmtCnnOp& op = d.cnn_ops[i];
      Gb.ch[i + 1] = op.kind == PMT_CNN_CONV ? op.out_ch : op.in_ch;
      Gb.len[i + 1] = op.out_len;
    }
    int off = 0, gmax = 0, stage = 4;
    for (int i = 0; i <= ns; ++i) {
      Gb.lp[i] = (Gb.len[i] + 3) & ~3;
      Gb.ld[i] = pad_ld(vt * Gb.lp[i]);
      Gb.act_off[i] = off;
      off += Gb.ch[i] * Gb.ld[i];
      if (Gb.ch[i] * Gb.ld[i] > gmax) gmax = Gb.ch[i] * Gb.ld[i];
    }
    for (int i = 0; i < ns; ++i) {
      const PmtCnnOp& op = d.cnn_ops[i];
      if (op.kind != PMT_CNN_CONV) continue;
      Gb.lpg[i] = (Gb.lp[i] + op.ksize - 1 + 3) & ~3;
      Gb.ldg[i] = pad_ld(vt * Gb.lpg[i]);
      if (i > 0 && op.out_ch * Gb.ldg[i] > gmax) gmax = op.out_ch * Gb.ldg[i];
      const int fwd = op.in_ch * op.ksize * ((op.out_ch + 7) / 8) * GROUP_STRIDE;
      const int bwd = op.out_ch * op.ksize * ((op.in_ch + 7) / 8) * GROUP_STRIDE;
      if (fwd > stage) stage = fwd;
      if (bwd > stage) stage = bwd;
    }
    int vs = Gb.ch[ns] * Gb.len[ns];
    for (int l = 0; l < Gb.n_linear; ++l) if (d.cnn_ops[ns + l].out_ch > vs) vs = d.cnn_ops[ns + l].out_ch;
    Gb.vs = (vs + 3) & ~3;
    Gb.act_total = (off + 3) & ~3;
    Gb.gbuf_floats = (gmax + 3) & ~3;
    Gb.stage_floats = (stage + 3) & ~3;
    smem = (size_t)(Gb.act_total + 2 * Gb.gbuf_floats + Gb.stage_floats + (Gb.n_linear + 3) * vt * Gb.vs + 16) * sizeof(float);
    if (smem <= 220 * 1024) break;
  }
  if (vt < 1) {
    *why = "haplotype CNN backward does not fit in shared memory";
    return false;
  }
  *smem_out = smem;
  return true;
}

static int launch_cnn_backward(const CallPlan& C, const float* weights, const float* image, const PmtBatch* batch,
                               const float* d_info_seq, float* partials, cudaStream_t st) {
  const CnnBwdGeom& Gb = C.cnn_bwd;
  const int B = batch->n_variants;
  int grid = (B + Gb.vt - 1) / Gb.vt;
  if (grid > PMT_PARTIAL_CTAS) grid = PMT_PARTIAL_CTAS;
  PMT_CUDA(cudaFuncSetAttribute(hap_cnn_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C.cnn_bwd_smem));
  hap_cnn_backward_kernel<<<grid, NTHREADS, C.cnn_bwd_smem, st>>>(C.P, C.G, Gb, weights, image + C.P.img_total, batch->haplotypes,
                                                                  batch->hap_kind, batch->hap_stride, B, d_info_seq, partials);
  return 0;
}

static size_t bwd_smem_bytes(const Plan& P) {
  const int n_head = P.d.d_feat + P.d.n_clusters * P.d.d_feat + 5 * P.d.n_clusters;
  const int acc_cap = n_head > 8 ? n_head : 8;
  return (size_t)(4 * P.bwd_rows * LD + 2 * P.stage_floats + 2 * TILE * 2 * P.sum_w + TILE * 2 * 16 + NWARPS * acc_cap +
                  64) * sizeof(float) + sizeof(HeadConst) + sizeof(TileMeta) + 64 + sizeof(Plan);
}
static int info_rows(const Plan& P) {
  int r = P.d.n_info_features;
  for (int i = 0; i < P.d.n_info_ops; ++i) if (P.d.info_ops[i].out_dim > r) r = P.d.info_ops[i].out_dim;
  return r;
}
// Claims go to CTAs round-robin (fixed summation order), so their number is a multiple of the grid; every claim ends with
// a partly filled tile, so a claim should hold >= 16 tiles (n_rows is an upper bound for a downsampled batch: claims of
// ~4 tiles left a fifth of the rows of every tile empty).
static Claims backward_claims(const PmtBatch* batch, int n_sm) {
  const int B = batch->n_variants;
  int per_cta = (int)((double)pmt_row_hint(batch) / ((double)n_sm * 16.0 * TILE));
  if (per_cta < 1) per_cta = 1;
  if (per_cta > 8) per_cta = 8;
  Claims K;
  K.claim = (int)((B + (long long)n_sm * per_cta - 1) / ((long long)n_sm * per_cta));
  if (K.claim < 1) K.claim = 1;
  K.n_claims = (B + K.claim - 1) / K.claim;
  K.grid = K.n_claims < PMT_PARTIAL_CTAS ? K.n_claims : PMT_PARTIAL_CTAS;
  if (K.grid > n_sm) K.grid = n_sm;
  return K;
}

void pmt_plan_backward(CallPlan& C, const PmtBatch* batch) {
  const Plan& P = C.P;
  C.bwd_smem = bwd_smem_bytes(P);
  C.info_bwd_smem = (size_t)(4 * info_rows(P) * LD + 2 * P.info_stage_floats) * sizeof(float);
  if (batch) C.bwd_claims = backward_claims(batch, C.n_sm);
  const char* cnn_why = nullptr;
  const bool cnn_ok = C.bwd_cnn_tc || cnn_bwd_simt_geom(P, C.G, &C.cnn_bwd, &C.cnn_bwd_smem, &cnn_why);
  char* why = C.bwd_refusal;
  const size_t n = sizeof(C.bwd_refusal);
  if (NPART * P.d.d_feat > P.bwd_rows)
    snprintf(why, n, "d_feat %d too wide for the backward kernel's head scratch", P.d.d_feat);
  else if (C.bwd_smem > 227 * 1024)
    snprintf(why, n, "model too wide for the backward kernel's shared-memory plan (%zu bytes)", C.bwd_smem);
  else if (C.info_bwd_smem > 227 * 1024)
    snprintf(why, n, "info MLP too wide for the backward kernel (%zu bytes of shared memory)", C.info_bwd_smem);
  else if (!cnn_ok)
    snprintf(why, n, "%s", cnn_why);
}
extern "C" int pmt_backward_kernels(const PmtModelDesc* desc, int32_t* reads_tc, int32_t* cnn_tc) {
  CallPlan C;
  if (pmt_call_plan(desc, nullptr, false, &C)) return 1;
  if (reads_tc) *reads_tc = C.bwd_reads_tc ? 1 : 0;
  if (cnn_tc) *cnn_tc = C.bwd_cnn_tc ? 1 : 0;
  return 0;
}

extern "C" int pmt_backward(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutGrads* grads,
                            float* d_weights, void* workspace, size_t workspace_bytes, void* stream) {
  CallPlan C;
  if (pmt_call_plan(desc, batch, false, &C)) return 1;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  BwdBuffers W;
  if (pmt_backward_buffers(C, workspace, workspace_bytes, &W)) return 1;
  PMT_CHECK(batch->n_variants > 0, "empty batch");
  PMT_CHECK(!C.bwd_refusal[0], "%s", C.bwd_refusal);

  const int B = batch->n_variants, w = desc->d_info + desc->d_seq;
  float* image = W.image;
  float* partials = W.partials;
  float* info_seq = W.info_seq;
  float* d_info_seq = W.d_info_seq;

  // what pmt_forward_train saved for this batch (PmtOutGrads.saved); the caller passes the buffer without its size
  SavedBuffers S;
  const bool saved = grads && grads->saved;
  if (saved) {
    PMT_CHECK(C.bwd_reads_tc && C.bwd_cnn_tc && C.mode == PMT_PRECISION_TF32X3 && grads->info_seq_be,
              "PmtOutGrads.saved needs the tf32x3 mode, the forward's info_seq_be, and the precision mode of the forward call");
    PMT_CHECK(C.saved.total > 0, "PmtOutGrads.saved: no saved-forward path for this batch");
    if (pmt_saved_buffers(C, grads->saved, C.saved.total, &S)) return 1;
  }
  PMT_CUDA(cudaMemsetAsync(partials, 0, C.bwd.partials.bytes, st));
  // conv images: only the SIMT haplotype-CNN kernels read them (the recompute below when the forward's embeddings are not
  // passed in, and the SIMT backward)
  pmt_launch_prepare(C, weights, image, st, true, !C.bwd_cnn_tc || !(grads && grads->info_seq_be));
  if (grads && grads->info_seq_be) {
    cudaMemcpyAsync(info_seq, grads->info_seq_be, (size_t)B * w * sizeof(float), cudaMemcpyDeviceToDevice, st);
  } else if (pmt_launch_info_mlp(C, weights, image, batch, info_seq, st) || pmt_launch_hap_cnn_simt(C, weights, image, batch, info_seq, st)) {
    return 1;
  }

  Plan P = C.P;
  P.claim_variants = C.bwd_claims.claim;
  const size_t smem = C.bwd_smem;

  BwdArgs A;
  A.wflat = weights; A.image = image; A.batch = *batch; A.info_seq = info_seq;
  A.d_logits_bk = grads ? grads->d_logits_bk : nullptr;
  A.d_alt_means = grads ? grads->d_alt_means_be : nullptr;
  A.d_ref_means = grads ? grads->d_ref_means_be : nullptr;
  A.d_info_seq = d_info_seq; A.scratch = W.scratch; A.scratch_stride = (long long)C.bwd.scr_floats; A.partials = partials;
  A.long_scratch = W.long_scratch; A.long_scratch_stride = (long long)C.bwd.long_floats;
  A.n_claims = C.bwd_claims.n_claims;
  int tc_grid = 0;
  if (C.bwd_reads_tc) {   // tile-sized sets; longer sets always take the SIMT long-set kernel
    if (pmt_launch_reads_tc_backward(C, weights, batch, info_seq, A.d_logits_bk, A.d_alt_means, A.d_ref_means, d_info_seq, W.tc,
                                     &tc_grid, st, saved ? &S : nullptr))
      return 1;
  } else {
    PMT_CUDA(cudaFuncSetAttribute(reads_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pmt_profile_begin(st);
    reads_backward_kernel<<<C.bwd_claims.grid, NTHREADS, smem, st>>>(P, A);
    pmt_profile_end(st);
  }
  if (C.bwd.long_grid > 0) {   // sets longer than a tile; same CTA-private gradient buffers, after the tile kernel: fixed order
    PMT_CUDA(cudaFuncSetAttribute(reads_backward_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    reads_backward_long_kernel<<<C.bwd.long_grid, NTHREADS, smem, st>>>(P, A);
  }
  {
    const size_t ismem = C.info_bwd_smem;
    const int n_tiles = (B + TILE - 1) / TILE;
    const int igrid = n_tiles < PMT_PARTIAL_CTAS ? n_tiles : PMT_PARTIAL_CTAS;
    PMT_CUDA(cudaFuncSetAttribute(info_mlp_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ismem));
    info_mlp_backward_kernel<<<igrid, NTHREADS, ismem, st>>>(P, weights, image, batch->info, batch->info_kind,
                                                             batch->info_stride, B, d_info_seq, W.scratch,
                                                             (long long)C.bwd.scr_floats, partials, info_rows(P));
  }
  if (C.bwd_cnn_tc) {
    if (pmt_launch_cnn_backward_mma(C, weights, batch, info_seq, d_info_seq, partials, W.cnn, st, saved ? S.cnn : nullptr)) return 1;
  } else if (launch_cnn_backward(C, weights, image, batch, d_info_seq, partials, st)) {
    return 1;
  }
  reduce_partials_kernel<<<(desc->n_params + 255) / 256, 256, 0, st>>>(partials, PMT_PARTIAL_CTAS, desc->n_params, d_weights);
  if (C.bwd_reads_tc && pmt_finish_reads_tc_backward(C, weights, d_weights, W.tc, tc_grid, st)) return 1;
  if (P.n_skipfix > 0) skip_fix_kernel<<<P.n_skipfix, 256, 0, st>>>(P, weights, d_weights);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_backward launch failed: %s", cudaGetErrorString(e));
  return 0;
}
