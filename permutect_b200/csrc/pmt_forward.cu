// Forward kernels of the ArtifactModel hot path (sm_100a) and the forward half of the C-ABI.
//
//   pack_weights_kernel   flat materialised weights -> GEMM-ready packed images        (once per call)
//   info_mlp_kernel       info_embedding MLP, one variant per row        (artifact_model.py:244)
//   hap_cnn_kernel        one-hot haplotypes + DNASequenceConvolution    (artifact_model.py:245, batch.py:115-130)
//   reads_forward_kernel  decode -> read_embedding -> concat -> gated ref/alt blocks -> reducer ->
//                         rotation -> clustering head -> per-variant sums (artifact_model.py:243-297)
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "pmt_call.h"
#include "pmt_tile.cuh"
#include "pmt_cnn.cuh"

namespace pmt {

// ------------------------------------------------------------------------------------------------
// weight packing
// ------------------------------------------------------------------------------------------------
__global__ void pack_weights_kernel(const __grid_constant__ Plan P, const float* __restrict__ w, float* __restrict__ image) {
  const GemmOp& op = P.gemm[blockIdx.x];
  const int per_image = op.K * op.G * GROUP_STRIDE;
  const int n_images = op.w_alt_off >= 0 ? 2 : 1;
  for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < per_image * n_images; idx += gridDim.y * blockDim.x) {
    const int which = idx / per_image, rem = idx % per_image;
    const int k = rem / (op.G * GROUP_STRIDE), slot = rem % (op.G * GROUP_STRIDE);
    const int grp = slot / GROUP_STRIDE, j = slot % GROUP_STRIDE;
    const int n = grp * op.NT + j;
    const int woff = which ? op.w_alt_off : op.w_off;
    image[op.img_off + idx] = (j < op.NT && n < op.N) ? w[woff + n * op.K + k] : 0.f;
  }
  // transposed image for the data-gradient GEMM: reduction over n (N rows), K outputs
  const int per_imageT = op.N * op.GT * GROUP_STRIDE;
  for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < per_imageT * n_images; idx += gridDim.y * blockDim.x) {
    const int which = idx / per_imageT, rem = idx % per_imageT;
    const int n = rem / (op.GT * GROUP_STRIDE), slot = rem % (op.GT * GROUP_STRIDE);
    const int grp = slot / GROUP_STRIDE, j = slot % GROUP_STRIDE;
    const int k = grp * op.NTT + j;
    const int woff = which ? op.w_alt_off : op.w_off;
    image[op.imgT_off + idx] = (j < op.NTT && k < op.K) ? w[woff + n * op.K + k] : 0.f;
  }
}

// conv weights [out][in][ks] -> image [(ci*ks + t)][G][8] with NT = 8
__global__ void pack_conv_kernel(const __grid_constant__ Plan P, const __grid_constant__ CnnGeom Gm,
                                 const float* __restrict__ w, float* __restrict__ image) {
  const PmtCnnOp& op = P.d.cnn_ops[blockIdx.x];
  if (op.kind != PMT_CNN_CONV) return;
  const int G = (op.out_ch + 7) / 8;
  const int total = op.in_ch * op.ksize * G * GROUP_STRIDE;
  float* img = image + Gm.img_off[blockIdx.x];
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int kk = idx / (G * GROUP_STRIDE), slot = idx % (G * GROUP_STRIDE);
    const int ci = kk / op.ksize, t = kk % op.ksize;
    const int co = (slot / GROUP_STRIDE) * 8 + slot % GROUP_STRIDE;
    img[idx] = co < op.out_ch ? w[op.w_off + (co * op.in_ch + ci) * op.ksize + t] : 0.f;
  }
}

// backward data gradient of a conv = convolution of dOut (zero-padded by ks-1) with the flipped kernel:
// image [(co*ks + t')][G over ci][8] = W[co][ci][ks-1-t']
__global__ void pack_convT_kernel(const __grid_constant__ Plan P, const __grid_constant__ CnnGeom Gm,
                                  const float* __restrict__ w, float* __restrict__ image) {
  const PmtCnnOp& op = P.d.cnn_ops[blockIdx.x];
  if (op.kind != PMT_CNN_CONV) return;
  const int G = (op.in_ch + 7) / 8;
  const int total = op.out_ch * op.ksize * G * GROUP_STRIDE;
  float* img = image + Gm.img_total + Gm.imgT_off[blockIdx.x];
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int kk = idx / (G * GROUP_STRIDE), slot = idx % (G * GROUP_STRIDE);
    const int co = kk / op.ksize, t = kk % op.ksize;
    const int ci = (slot / GROUP_STRIDE) * 8 + slot % GROUP_STRIDE;
    img[idx] = ci < op.in_ch ? w[op.w_off + (co * op.in_ch + ci) * op.ksize + (op.ksize - 1 - t)] : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------
// info MLP: rows of the tile are variants
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NTHREADS, 1)
info_mlp_kernel(const __grid_constant__ Plan P, const float* __restrict__ wflat, const float* __restrict__ image,
                const void* __restrict__ info, int info_kind, long long info_stride, int n_variants,
                float* __restrict__ info_seq) {
  extern __shared__ __align__(16) float smem[];
  const int in_rows = P.d.n_info_features > PMT_MAX_DIM ? PMT_MAX_INFO_DIM : PMT_MAX_DIM;
  float* b0 = smem;                       // input buffer (up to 128 features)
  float* b1 = b0 + in_rows * LD;
  float* b2 = b1 + PMT_MAX_DIM * LD;
  float* st0 = b2 + PMT_MAX_DIM * LD;
  float* st1 = st0 + P.info_stage_floats;
  Stage stage;
  stage.init(st0, st1, image, &P);
  const int v0 = blockIdx.x * TILE;
  const int nv = min(TILE, n_variants - v0);
  const int I = P.d.n_info_features;
  stage.prefetch(P.info_g0);
  for (int idx = threadIdx.x; idx < TILE * I; idx += NTHREADS) {
    const int r = idx / I, f = idx % I;
    float v = 0.f;
    if (r < nv) {
      const long long off = (long long)(v0 + r) * info_stride + f;
      v = info_kind == PMT_F16 ? __half2float(reinterpret_cast<const __half*>(info)[off])
                               : reinterpret_cast<const float*>(info)[off];
    }
    b0[f * LD + r] = v;
  }
  float* out = run_mlp(P, P.d.info_ops, P.d.n_info_ops, P.info_g0, b0, b1, b2, b0, stage, wflat, TILE, -1);
  __syncthreads();
  const int w = P.d.d_info + P.d.d_seq;
  for (int idx = threadIdx.x; idx < nv * P.d.d_info; idx += NTHREADS) {
    const int r = idx / P.d.d_info, j = idx % P.d.d_info;
    info_seq[(long long)(v0 + r) * w + j] = out[j * LD + r];
  }
}

// ------------------------------------------------------------------------------------------------
// info_embedding MLP, one THREAD per variant (artifact_model.py:244; mlp.py:8-76).  The whole MLP is ~4 k multiply-adds
// per variant on vectors of d_info (20) numbers: a tile GEMM spends its time in barriers and weight staging, so here the
// weights of every layer sit in shared memory for the life of the CTA ([k][W] rows: one broadcast 16-byte load feeds four
// multiply-adds), a thread keeps the running vector, the DenseSkipBlock residual and the layer output in registers, and
// the input block of a tile is staged feature-major through shared memory with coalesced loads.
// W4 = ceil(widest hidden vector / 4); layers after the first have in_dim <= 4 * W4.
// ------------------------------------------------------------------------------------------------
constexpr int INFO_TPB = 128;
template <int W4>
__global__ void __launch_bounds__(INFO_TPB)
info_mlp_rows_kernel(const __grid_constant__ PmtModelDesc D, const float* __restrict__ wflat, const void* __restrict__ info, int info_kind,
                     long long info_stride, int n_variants, float* __restrict__ info_seq) {
  constexpr int W = 4 * W4;
  extern __shared__ __align__(16) float smem[];
  const int I = D.n_info_features, n_ops = D.n_info_ops;
  // carve: per op [in_dim][W] transposed weights + [W] bias, then the input tile [I][INFO_TPB + 1]
  float* wt = smem;
  int off = 0;
  for (int i = 0; i < n_ops; ++i) off += (D.info_ops[i].in_dim + 1) * W;
  float* sx = smem + off;
  {
    int base = 0;
    for (int i = 0; i < n_ops; ++i) {
      const PmtLinearOp& op = D.info_ops[i];
      for (int idx = threadIdx.x; idx < (op.in_dim + 1) * W; idx += INFO_TPB) {
        const int k = idx / W, n = idx - k * W;
        float v = 0.f;
        if (n < op.out_dim) v = k < op.in_dim ? __ldg(wflat + op.w_off + n * op.in_dim + k) : __ldg(wflat + op.b_off + n);
        wt[base + idx] = v;
      }
      base += (op.in_dim + 1) * W;
    }
  }
  const int out_w = D.d_info + D.d_seq;
  const int n_tiles = (n_variants + INFO_TPB - 1) / INFO_TPB;
  const int r = threadIdx.x;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int v0 = tile * INFO_TPB, nv = min(INFO_TPB, n_variants - v0);
    __syncthreads();   // weights staged / previous tile's readers done
    const bool raw16 = info_kind == PMT_F16 && info_stride >= I && info_stride <= I + 8 && (reinterpret_cast<uintptr_t>(info) & 3) == 0;
    if (raw16) {
      // fp16 rows a few columns apart (the float array of the dataset): the tile's rows are one contiguous span, copied as
      // 32-bit words; every thread then converts its own row
      const unsigned* src = reinterpret_cast<const unsigned*>(reinterpret_cast<const __half*>(info) + (long long)v0 * info_stride);
      unsigned* raw = reinterpret_cast<unsigned*>(sx);
      const int n_halves = (int)((nv - 1) * info_stride) + I;     // up to the last row's last feature, not a byte further
      const int n_words = n_halves >> 1;
      for (int idx = threadIdx.x; idx < n_words; idx += INFO_TPB) raw[idx] = __ldg(src + idx);
      if ((n_halves & 1) && threadIdx.x == 0)
        reinterpret_cast<__half*>(sx)[n_halves - 1] = __ldg(reinterpret_cast<const __half*>(src) + n_halves - 1);
    } else {
      for (int idx = threadIdx.x; idx < nv * I; idx += INFO_TPB) {
        const int rr = idx / I, f = idx - rr * I;
        const long long o = (long long)(v0 + rr) * info_stride + f;
        sx[f * (INFO_TPB + 1) + rr] = info_kind == PMT_F16 ? __half2float(__ldg(reinterpret_cast<const __half*>(info) + o))
                                                            : __ldg(reinterpret_cast<const float*>(info) + o);
      }
    }
    __syncthreads();
    if (r >= nv) continue;
    float cur[W], res[W];
#pragma unroll
    for (int n = 0; n < W; ++n) { cur[n] = 0.f; res[n] = 0.f; }
    int base = 0;
    for (int i = 0; i < n_ops; ++i) {
      const PmtLinearOp op = D.info_ops[i];
      const float* w = wt + base;
      float y[W];
      {
        const float4* b4 = reinterpret_cast<const float4*>(w + op.in_dim * W);
#pragma unroll
        for (int q = 0; q < W4; ++q) { const float4 b = b4[q]; y[4 * q] = b.x; y[4 * q + 1] = b.y; y[4 * q + 2] = b.z; y[4 * q + 3] = b.w; }
      }
      if (i == 0) {   // input layer: the staged tile (raw fp16 rows, or feature-major floats)
        const float* xr = sx + r;
        const __half* hr = reinterpret_cast<const __half*>(sx) + (long long)r * info_stride;
#pragma unroll 4
        for (int k = 0; k < op.in_dim; ++k) {
          const float x = raw16 ? __half2float(hr[k]) : xr[k * (INFO_TPB + 1)];
          const float4* w4 = reinterpret_cast<const float4*>(w + k * W);
#pragma unroll
          for (int q = 0; q < W4; ++q) {
            const float4 ww = w4[q];
            y[4 * q] = fmaf(x, ww.x, y[4 * q]); y[4 * q + 1] = fmaf(x, ww.y, y[4 * q + 1]);
            y[4 * q + 2] = fmaf(x, ww.z, y[4 * q + 2]); y[4 * q + 3] = fmaf(x, ww.w, y[4 * q + 3]);
          }
        }
      } else {
        float src[W];
        if (op.flags & PMT_OP_SKIP_BEGIN) {
#pragma unroll
          for (int n = 0; n < W; ++n) { res[n] = cur[n]; src[n] = selu(cur[n]); }
        } else {
#pragma unroll
          for (int n = 0; n < W; ++n) src[n] = cur[n];
        }
#pragma unroll
        for (int k = 0; k < W; ++k) {
          if (k < op.in_dim) {
            const float x = src[k];
            const float4* w4 = reinterpret_cast<const float4*>(w + k * W);
#pragma unroll
            for (int q = 0; q < W4; ++q) {
              const float4 ww = w4[q];
              y[4 * q] = fmaf(x, ww.x, y[4 * q]); y[4 * q + 1] = fmaf(x, ww.y, y[4 * q + 1]);
              y[4 * q + 2] = fmaf(x, ww.z, y[4 * q + 2]); y[4 * q + 3] = fmaf(x, ww.w, y[4 * q + 3]);
            }
          }
        }
      }
      if (op.flags & PMT_OP_SKIP_END) {
        const float alpha = __ldg(wflat + op.alpha_off);
#pragma unroll
        for (int n = 0; n < W; ++n) cur[n] = fmaf(alpha, y[n], res[n]);
      } else if (op.flags & PMT_OP_POST_SELU) {
#pragma unroll
        for (int n = 0; n < W; ++n) cur[n] = n < op.out_dim ? selu(y[n]) : 0.f;
      } else {
#pragma unroll
        for (int n = 0; n < W; ++n) cur[n] = y[n];
      }
      base += (op.in_dim + 1) * W;
    }
    float* dst = info_seq + (long long)(v0 + r) * out_w;
#pragma unroll
    for (int n = 0; n < W; ++n) if (n < D.d_info) dst[n] = cur[n];
  }
}

// Small batches: the thread-per-variant kernel above is a chain of ~7 600 dependent multiply-adds per variant (30 us for the 64
// variants of the reference's default batch, a quarter of the whole inference call).  Here a WARP owns a variant and a lane
// owns one output of every layer: the chain is in_dim FMAs long per layer, inputs travel by shuffle.  Same order of
// summation (bias first, inputs in ascending order), so the results are bitwise those of the other kernel.
constexpr int INFO_WARPS = 8;
__global__ void __launch_bounds__(32 * INFO_WARPS)
info_mlp_warp_kernel(const __grid_constant__ PmtModelDesc D, const float* __restrict__ wflat, const void* __restrict__ info, int info_kind,
                     long long info_stride, int n_variants, float* __restrict__ info_seq) {
  constexpr int W = 32;
  extern __shared__ __align__(16) float smem[];
  const int I = D.n_info_features, n_ops = D.n_info_ops;
  float* wt = smem;   // per op [in_dim + 1][W]: transposed weights, then the bias row
  {
    // zero (the padding outputs), then the weights read in the order they lie in memory (coalesced) and transposed on the
    // way into shared memory: at this batch size the staging is a good part of the kernel
    int total = 0;
    for (int i = 0; i < n_ops; ++i) total += (D.info_ops[i].in_dim + 1) * W;
    for (int idx = threadIdx.x; idx < total; idx += 32 * INFO_WARPS) wt[idx] = 0.f;
    __syncthreads();
    int base = 0;
    for (int i = 0; i < n_ops; ++i) {
      const PmtLinearOp& op = D.info_ops[i];
      const int nk = op.out_dim * op.in_dim;
      for (int idx = threadIdx.x; idx < nk + op.out_dim; idx += 32 * INFO_WARPS) {
        if (idx < nk) {
          const int n = idx / op.in_dim, k = idx - n * op.in_dim;
          wt[base + k * W + n] = __ldg(wflat + op.w_off + idx);
        } else {
          wt[base + op.in_dim * W + (idx - nk)] = __ldg(wflat + op.b_off + idx - nk);
        }
      }
      base += (op.in_dim + 1) * W;
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int out_w = D.d_info + D.d_seq;
  for (int v = blockIdx.x * INFO_WARPS + warp; v < n_variants; v += gridDim.x * INFO_WARPS) {
    // the variant's features, lane l holding features l, l + 32, ...
    float xin[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int f = q * 32 + lane;
      float x = 0.f;
      if (f < I) {
        const long long o = (long long)v * info_stride + f;
        x = info_kind == PMT_F16 ? __half2float(__ldg(reinterpret_cast<const __half*>(info) + o)) : __ldg(reinterpret_cast<const float*>(info) + o);
      }
      xin[q] = x;
    }
    float cur = 0.f, res = 0.f;
    int base = 0;
    for (int i = 0; i < n_ops; ++i) {
      const PmtLinearOp op = D.info_ops[i];
      const float* w = wt + base + lane;
      float y = w[op.in_dim * W];   // bias
      if (i == 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          if (q * 32 < op.in_dim) {
            const int kn = min(32, op.in_dim - q * 32);
            for (int k = 0; k < kn; ++k) y = fmaf(__shfl_sync(0xffffffffu, xin[q], k), w[(q * 32 + k) * W], y);
          }
        }
      } else {
        float src = cur;
        if (op.flags & PMT_OP_SKIP_BEGIN) { res = cur; src = selu(cur); }
        for (int k = 0; k < op.in_dim; ++k) y = fmaf(__shfl_sync(0xffffffffu, src, k), w[k * W], y);
      }
      if (op.flags & PMT_OP_SKIP_END) cur = fmaf(__ldg(wflat + op.alpha_off), y, res);
      else if (op.flags & PMT_OP_POST_SELU) cur = lane < op.out_dim ? selu(y) : 0.f;
      else cur = y;
      base += (op.in_dim + 1) * W;
    }
    if (lane < D.d_info) info_seq[(long long)v * out_w + lane] = cur;
  }
}

// The thread-per-variant kernel covers MLPs whose hidden vectors are at most 32 wide, with the input layer first and no
// DenseSkipBlock opening on the raw input; anything else takes the tile-GEMM kernel above.
static int info_rows_w4(const PmtModelDesc& d) {
  if (d.n_info_ops < 1 || d.n_info_features > 256) return 0;
  int widest = 0;
  for (int i = 0; i < d.n_info_ops; ++i) {
    const PmtLinearOp& op = d.info_ops[i];
    if (op.out_dim > widest) widest = op.out_dim;
    if (i > 0 && op.in_dim > widest) return 0;
    if (i == 0 && (op.flags & (PMT_OP_SKIP_BEGIN | PMT_OP_SKIP_END))) return 0;
    if (i == 0 && op.in_dim != d.n_info_features) return 0;
  }
  if (d.info_ops[d.n_info_ops - 1].out_dim != d.d_info) return 0;
  const int w4 = (widest + 3) / 4;
  return (w4 >= 1 && w4 <= 8) ? w4 : 0;
}

template <int W4>
static int launch_info_rows(const PmtModelDesc& d, const float* weights, const PmtBatch* batch, float* info_seq, size_t smem,
                            cudaStream_t st) {
  PMT_CUDA(cudaFuncSetAttribute(info_mlp_rows_kernel<W4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int n_tiles = (batch->n_variants + INFO_TPB - 1) / INFO_TPB;
  int per_sm = (int)((220 * 1024) / smem);
  if (per_sm > 8) per_sm = 8;
  if (per_sm < 1) per_sm = 1;
  const int grid = n_tiles < 148 * per_sm ? n_tiles : 148 * per_sm;
  info_mlp_rows_kernel<W4><<<grid, INFO_TPB, smem, st>>>(d, weights, batch->info, batch->info_kind, batch->info_stride, batch->n_variants, info_seq);
  return 0;
}

// ------------------------------------------------------------------------------------------------
// haplotype CNN
// ------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(NTHREADS, 1)
hap_cnn_kernel(const __grid_constant__ Plan P, const __grid_constant__ CnnGeom Gm, const float* __restrict__ wflat,
               const float* __restrict__ conv_image, const void* __restrict__ haps, int hap_kind, long long hap_stride,
               int n_variants, float* __restrict__ info_seq) {
  extern __shared__ __align__(16) float smem[];
  float* bufA = smem;
  float* bufB = bufA + Gm.buf_floats;
  float* wimg = bufB + Gm.buf_floats;
  float* vec0 = wimg + Gm.img_total;  // [vt][256] linear-stack scratch
  float* vec1 = vec0 + Gm.vt * 256;
  for (int i = threadIdx.x; i < Gm.img_total / 4; i += NTHREADS)
    reinterpret_cast<float4*>(wimg)[i] = __ldg(reinterpret_cast<const float4*>(conv_image) + i);
  for (int i = threadIdx.x; i < 2 * Gm.buf_floats; i += NTHREADS) bufA[i] = 0.f;
  __syncthreads();
  const int L = P.d.hap_len;
  const int vt = Gm.vt;
  const int out_w = P.d.d_info + P.d.d_seq;
  for (int v0 = blockIdx.x * vt; v0 < n_variants; v0 += gridDim.x * vt) {
    const int nv = min(vt, n_variants - v0);
    // one-hot input, batch.py:115-130: channel 2c + h is "haplotype h (0 ref, 1 alt) has code c at position p"
    const int ld0 = vt * Gm.lp[0] + 8;
    for (int idx = threadIdx.x; idx < nv * 2 * L; idx += NTHREADS) {
      const int v = idx / (2 * L), hp = idx % (2 * L);
      const long long off = (long long)(v0 + v) * hap_stride + hp;
      const int code = hap_kind == PMT_I64 ? (int)reinterpret_cast<const long long*>(haps)[off]
                                           : (int)reinterpret_cast<const short*>(haps)[off];
      const int h = hp / L, p = hp % L;
#pragma unroll
      for (int c = 0; c < 5; ++c) bufA[(2 * c + h) * ld0 + v * Gm.lp[0] + p] = (code == c) ? 1.f : 0.f;
    }
    __syncthreads();
    float* in = bufA;
    float* out = bufB;
    int i = 0;
    for (; i < Gm.n_spatial; ++i) {
      const PmtCnnOp& op = P.d.cnn_ops[i];
      const int in_ld = vt * Gm.lp[i] + 8, out_ld = vt * Gm.lp[i + 1] + 8;
      if (op.kind == PMT_CNN_CONV) {
        const float* img = wimg + Gm.img_off[i];
        PMT_CONV_DISPATCH(op.ksize, op, in, in_ld, Gm.lp[i], out, out_ld, Gm.lp[i + 1], img, wflat, vt)
      } else {  // max pool, dna_sequence_convolution.py:75-77
        const int total = op.in_ch * vt * op.out_len;
        for (int idx = threadIdx.x; idx < total; idx += NTHREADS) {
          const int c = idx / (vt * op.out_len), rem = idx % (vt * op.out_len);
          const int v = rem / op.out_len, p = rem % op.out_len;
          const float* src = in + c * in_ld + v * Gm.lp[i] + p * op.stride;
          float m = src[0];
          for (int t = 1; t < op.ksize; ++t) m = fmaxf(m, src[t]);
          out[c * out_ld + v * Gm.lp[i + 1] + p] = m;
        }
      }
      __syncthreads();
      float* tmp = in; in = out; out = tmp;
    }
    // flatten (channel-major, dna_sequence_convolution.py:84-89) + linear stack
    {
      const PmtCnnOp& last = P.d.cnn_ops[Gm.n_spatial - 1];
      const int C = Gm.n_spatial > 0 ? (last.kind == PMT_CNN_CONV ? last.out_ch : last.in_ch) : 10;
      const int len = Gm.n_spatial > 0 ? last.out_len : L;
      const int in_ld = vt * Gm.lp[Gm.n_spatial] + 8;
      const float* vin = nullptr;
      float* vout = vec0;
      for (; i < P.d.n_cnn_ops; ++i) {
        const PmtCnnOp& op = P.d.cnn_ops[i];
        const bool is_last = (i + 1 == P.d.n_cnn_ops);
        for (int idx = threadIdx.x; idx < nv * op.out_ch; idx += NTHREADS) {
          const int v = idx / op.out_ch, n = idx % op.out_ch;
          float acc = __ldg(wflat + op.b_off + n);
          const float* wr = wflat + op.w_off + (long long)n * op.in_ch;
          if (vin == nullptr) {
            for (int c = 0; c < C; ++c)
              for (int p = 0; p < len; ++p) acc = fmaf(__ldg(wr + c * len + p), in[c * in_ld + v * Gm.lp[Gm.n_spatial] + p], acc);
          } else {
            for (int k = 0; k < op.in_ch; ++k) acc = fmaf(__ldg(wr + k), vin[v * 256 + k], acc);
          }
          acc = apply_act(acc, op.act);
          if (is_last) info_seq[(long long)(v0 + v) * out_w + P.d.d_info + n] = acc;
          else vout[v * 256 + n] = acc;
        }
        __syncthreads();
        vin = vout;
        vout = (vout == vec0) ? vec1 : vec0;
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// read path
// ------------------------------------------------------------------------------------------------
// Variants whose reads fit one tile (the only case on real data: reads are capped at 10 ref + 15 alt at
// ingest, plain_text_data.py:172-174).  Persistent CTAs claim runs of variants from an atomic counter and
// pack them greedily into tiles; everything between the compressed reads and the per-variant outputs
// stays in shared memory.
__global__ void __launch_bounds__(NTHREADS, 1)
reads_forward_kernel(const __grid_constant__ Plan P, const __grid_constant__ ReadKernelArgs A) {
  extern __shared__ __align__(16) float smem[];
  const PmtModelDesc& D = P.d;
  TileCtx C;
  float *st0, *st1;
  carve_tile_ctx(P, smem, C, st0, st1, P.stage_floats);
  C.W = A.wflat;
  __shared__ int s_claim;
  const int tid = threadIdx.x;
  const int B = A.batch.n_variants;
  Stage stage;
  stage.init(st0, st1, A.image, &P);
  if (tid == 0) head_constants(D, C.W, C.HC);
  for (int i = tid; i < 3 * PMT_MAX_DIM * LD; i += NTHREADS) C.X[i] = 0.f;
  __syncthreads();
  const long long total_ref = __ldg(A.batch.ref_off + B);  // == sum of ref counts
  const int claim = P.claim_variants;

  for (;;) {
    if (tid == 0) s_claim = atomicAdd(A.claim_counter, 1);
    __syncthreads();
    const long long cv0 = (long long)s_claim * claim;
    __syncthreads();
    if (cv0 >= B) break;
    const int cv1 = (int)min((long long)B, cv0 + claim);
    int v_cur = (int)cv0;
    while (v_cur < cv1) {
      const int nv = build_tile(A.batch, v_cur, cv1, total_ref, *C.M);
      if (nv == 0) { v_cur += 1; continue; }   // longer than a tile: handled by reads_forward_long_kernel
      v_cur += nv;
      C.rows_used = (C.M->rows + 3) & ~3;
      tile_embed(P, C, stage, A.batch, A.out.info_seq_be, nullptr);
      for (int blk = 0; blk < D.n_blocks; ++blk) {
        block_phase_a(P, C, stage, blk, nullptr);
        segment_sums(*C.M, C.T2, D.d_ffn / 2, D.d_ffn / 2, C.sums, P.sum_w, false, false);
        __syncthreads();
        block_means(P, C, blk);
        block_phase_b(P, C, stage, blk, blk + 1 < D.n_blocks ? P.blk_g0 + 2 * blk + 2 : P.red_g0);
      }
      float *y, *Fb;
      tile_tail(P, C, stage, A.out, false, nullptr, y, Fb);
      tile_outputs(P, C, A.out);
      __syncthreads();
    }
  }
}

// Variants with more reads than a tile (synthetic high-depth sets, BASELINE config 5).  One CTA walks the
// variant in chunks of TILE rows; the residual stream x and the gated-block hidden z of every chunk live
// in a per-CTA global scratch (L2 resident for moderately long sets); the per-block mean fields and the
// final sums are accumulated across chunks, which is the only cross-read coupling (gated_mlp.py:236-248).
__global__ void __launch_bounds__(NTHREADS, 1)
reads_forward_long_kernel(const __grid_constant__ Plan P, const __grid_constant__ ReadKernelArgs A) {
  extern __shared__ __align__(16) float smem[];
  const PmtModelDesc& D = P.d;
  TileCtx C;
  float *st0, *st1;
  carve_tile_ctx(P, smem, C, st0, st1, P.stage_floats);
  C.W = A.wflat;
  const int tid = threadIdx.x;
  const int B = A.batch.n_variants;
  Stage stage;
  stage.init(st0, st1, A.image, &P);
  if (tid == 0) head_constants(D, C.W, C.HC);
  for (int i = tid; i < 3 * PMT_MAX_DIM * LD; i += NTHREADS) C.X[i] = 0.f;
  __syncthreads();
  const long long total_ref = __ldg(A.batch.ref_off + B);
  float* scr = A.scratch + (long long)blockIdx.x * A.scratch_stride;
  const int x_img = D.d_model * LD, z_img = D.d_ffn * LD, chunk_img = x_img + z_img;
  const int H = D.d_ffn / 2;

  for (int v = blockIdx.x; v < B; v += gridDim.x) {
    const long long nref = __ldg(A.batch.ref_off + v + 1) - __ldg(A.batch.ref_off + v);
    const long long nalt = __ldg(A.batch.alt_off + v + 1) - __ldg(A.batch.alt_off + v);
    const long long total = ((nref + 3) & ~3LL) + nalt;
    if (total <= TILE) continue;
    const int n_chunks = (int)((total + TILE - 1) / TILE);
    for (int c = 0; c < n_chunks; ++c) {
      build_chunk(A.batch, v, c, total_ref, *C.M);
      C.rows_used = (C.M->rows + 3) & ~3;
      tile_embed(P, C, stage, A.batch, A.out.info_seq_be, nullptr);
      save_rows(C.X, D.d_model, scr + (long long)c * chunk_img);
      __syncthreads();
    }
    for (int blk = 0; blk < D.n_blocks; ++blk) {
      for (int c = 0; c < n_chunks; ++c) {
        build_chunk(A.batch, v, c, total_ref, *C.M);
        C.rows_used = (C.M->rows + 3) & ~3;
        load_rows(C.X, D.d_model, scr + (long long)c * chunk_img);
        __syncthreads();
        block_phase_a(P, C, stage, blk, nullptr);
        save_rows(C.T2, D.d_ffn, scr + (long long)c * chunk_img + x_img);   // z1 and the normalised z2
        segment_sums(*C.M, C.T2, H, H, C.sums, P.sum_w, false, c > 0);
        __syncthreads();
      }
      block_means(P, C, blk);
      for (int c = 0; c < n_chunks; ++c) {
        build_chunk(A.batch, v, c, total_ref, *C.M);
        C.rows_used = (C.M->rows + 3) & ~3;
        load_rows(C.X, D.d_model, scr + (long long)c * chunk_img);
        load_rows(C.T2, D.d_ffn, scr + (long long)c * chunk_img + x_img);
        __syncthreads();
        block_phase_b(P, C, stage, blk, -1);
        save_rows(C.X, D.d_model, scr + (long long)c * chunk_img);
        __syncthreads();
      }
    }
    for (int c = 0; c < n_chunks; ++c) {
      build_chunk(A.batch, v, c, total_ref, *C.M);
      C.rows_used = (C.M->rows + 3) & ~3;
      load_rows(C.X, D.d_model, scr + (long long)c * chunk_img);
      __syncthreads();
      float *y, *Fb;
      tile_tail(P, C, stage, A.out, c > 0, nullptr, y, Fb);
    }
    tile_outputs(P, C, A.out);
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// stand-alone decode (Batch.__init__, batch.py:51-56)
// ------------------------------------------------------------------------------------------------
__global__ void decode_reads_kernel(const uint8_t* __restrict__ reads, long long n_rows, int row_bytes, float* __restrict__ out) {
  const int F = 56 + row_bytes - 7;
  const long long total = n_rows * F;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx / F;
    const int f = (int)(idx % F);
    const uint8_t* rp = reads + r * row_bytes;
    float v;
    if (f < 56) v = (float)((rp[f >> 3] >> (7 - (f & 7))) & 1u);
    else v = (float)((rp[7 + f - 56] + 128u) & 255u) * 0.03125f;
    out[idx] = v;
  }
}

}  // namespace pmt

// ================================================================================================
// host side
// ================================================================================================
using namespace pmt;

static thread_local char g_err[512] = "";
void pmt_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* pmt_last_error(void) { return g_err; }
// process-wide on purpose: autograd runs pmt_backward on its own host thread
static cudaEvent_t g_prof_start = nullptr, g_prof_stop = nullptr;
extern "C" int pmt_set_profile_events(void* start_event, void* stop_event) {
  g_prof_start = reinterpret_cast<cudaEvent_t>(start_event);
  g_prof_stop = reinterpret_cast<cudaEvent_t>(stop_event);
  return 0;
}
void pmt_profile_begin(cudaStream_t st) { if (g_prof_start && g_prof_stop) cudaEventRecord(g_prof_start, st); }
void pmt_profile_end(cudaStream_t st) { if (g_prof_start && g_prof_stop) cudaEventRecord(g_prof_stop, st); }
extern "C" int pmt_abi_version(void) { return PMT_ABI_VERSION; }

// Column groups of a tile GEMM: one warp per group, so eight groups keep all eight warps busy (four groups for N <= 32
// left half the CTA at the barrier: 22.7 -> 21.4 ms on the backward kernel).
static void choose_groups(int N, int* G, int* NT) {
  int nt = (N + 7) / 8;
  if (nt == 3) nt = 4;   // N = 20: five groups of four instead of seven of three (a third less staged image, 8 floats per group)
  if (nt < 1) nt = 1;
  *G = (N + nt - 1) / nt;
  *NT = nt;
}

static int add_gemm(Plan& P, int K, int N, int w, int b, int w_alt, int b_alt) {
  if (P.n_gemm >= MAX_GEMM) return -1;
  GemmOp& op = P.gemm[P.n_gemm];
  op.K = K; op.N = N;
  choose_groups(N, &op.G, &op.NT);
  op.w_off = w; op.b_off = b; op.w_alt_off = w_alt; op.b_alt_off = b_alt;
  op.img_off = P.img_total;
  op.img_floats = K * op.G * GROUP_STRIDE * (w_alt >= 0 ? 2 : 1);
  op.img_floats = (op.img_floats + 3) & ~3;
  P.img_total += op.img_floats;
  choose_groups(K, &op.GT, &op.NTT);
  op.imgT_off = P.img_total;
  op.imgT_floats = (N * op.GT * GROUP_STRIDE * (w_alt >= 0 ? 2 : 1) + 3) & ~3;
  P.img_total += op.imgT_floats;
  return P.n_gemm++;
}

int pmt_build_plan(const PmtModelDesc* d, Plan* out) {
  Plan& P = *out;
  memset(&P, 0, sizeof(P));
  if (d->abi_version != PMT_ABI_VERSION) { pmt_set_error("PmtModelDesc.abi_version %d != %d", d->abi_version, PMT_ABI_VERSION); return 1; }
  P.d = *d;
  PMT_CHECK(d->n_read_features <= PMT_MAX_DIM && d->n_read_features == 56 + d->read_row_bytes - 7,
            "n_read_features %d unsupported (max %d, must equal 8*7 + row_bytes - 7)", d->n_read_features, PMT_MAX_DIM);
  PMT_CHECK(d->n_info_features <= PMT_MAX_INFO_DIM, "n_info_features %d > %d", d->n_info_features, PMT_MAX_INFO_DIM);
  PMT_CHECK(d->d_model <= PMT_MAX_DIM && d->d_model == d->d_read + d->d_info + d->d_seq, "d_model %d unsupported", d->d_model);
  PMT_CHECK(d->d_ffn <= PMT_MAX_DIM && d->d_ffn % 2 == 0, "d_ffn %d unsupported", d->d_ffn);
  // d_ffn 2: the spatial gating unit's LayerNorm sees one feature and outputs its bias whatever the input, so the ref reads
  // never reach the loss and the gradients through that LayerNorm are rounding noise scaled by 1 / sqrt(eps)
  PMT_CHECK(d->d_ffn >= 4, "d_ffn %d: self_attention_hidden_dimension must be at least 4 (a one-feature spatial gating unit "
            "is constant)", d->d_ffn);
  PMT_CHECK(d->d_feat <= PMT_MAX_FEAT && d->n_clusters <= PMT_MAX_CLUSTERS && d->n_clusters >= 1, "d_feat/n_clusters unsupported");
  PMT_CHECK(d->n_blocks <= PMT_MAX_BLOCKS, "too many gated blocks");
  PMT_CHECK(d->n_read_ops <= PMT_MAX_MLP_OPS && d->n_info_ops <= PMT_MAX_MLP_OPS && d->n_red_ops <= PMT_MAX_MLP_OPS &&
            d->n_cnn_ops <= PMT_MAX_CNN_OPS, "too many layers");
  auto add_program = [&](const PmtLinearOp* ops, int n, int max_in, int* g0) -> int {
    *g0 = P.n_gemm;
    for (int i = 0; i < n; ++i) {
      if (ops[i].in_dim > (i == 0 ? max_in : PMT_MAX_DIM) || ops[i].out_dim > PMT_MAX_DIM) { pmt_set_error("layer width > %d", PMT_MAX_DIM); return 1; }
      if (add_gemm(P, ops[i].in_dim, ops[i].out_dim, ops[i].w_off, ops[i].b_off, -1, -1) < 0) { pmt_set_error("too many GEMMs"); return 1; }
    }
    return 0;
  };
  if (add_program(d->read_ops, d->n_read_ops, PMT_MAX_DIM, &P.read_g0)) return 1;
  P.blk_g0 = P.n_gemm;
  for (int b = 0; b < d->n_blocks; ++b) {
    const PmtBlockOffsets& o = d->blocks[b];
    add_gemm(P, d->d_model, d->d_ffn, o.p1_ref_w, o.p1_ref_b, o.p1_alt_w, o.p1_alt_b);
    add_gemm(P, d->d_ffn / 2, d->d_model, o.p2_ref_w, o.p2_ref_b, o.p2_alt_w, o.p2_alt_b);
  }
  if (add_program(d->red_ops, d->n_red_ops, PMT_MAX_DIM, &P.red_g0)) return 1;
  int read_path_end = P.n_gemm;
  if (add_program(d->info_ops, d->n_info_ops, PMT_MAX_INFO_DIM, &P.info_g0)) return 1;
  for (int g = 0; g < P.n_gemm; ++g) {
    int& tgt = g < read_path_end ? P.stage_floats : P.info_stage_floats;
    if (P.gemm[g].img_floats > tgt) tgt = P.gemm[g].img_floats;
    if (P.gemm[g].imgT_floats > tgt) tgt = P.gemm[g].imgT_floats;
  }
  P.sum_w = d->d_ffn / 2 > d->d_feat ? d->d_ffn / 2 : d->d_feat;
  P.claim_variants = 64;
  // backward: activation scratch layout, buffer height, DenseSkipBlock fix-ups
  int off = 0, rows = d->d_model;
  auto grow = [&](int v) { if (v > rows) rows = v; };
  for (int i = 0; i < d->n_read_ops; ++i) { P.scr_read[i] = off; off += d->read_ops[i].in_dim * LD; grow(d->read_ops[i].in_dim); grow(d->read_ops[i].out_dim); }
  for (int b = 0; b < d->n_blocks; ++b) { P.scr_x[b] = off; off += d->d_model * LD; P.scr_z[b] = off; off += d->d_ffn * LD; }
  for (int i = 0; i < d->n_red_ops; ++i) { P.scr_red[i] = off; off += d->red_ops[i].in_dim * LD; grow(d->red_ops[i].in_dim); grow(d->red_ops[i].out_dim); }
  P.scr_red[d->n_red_ops] = off; off += d->d_feat * LD;
  P.scratch_floats = off;
  grow(3 * d->d_ffn); grow(d->d_feat + d->n_clusters + 2);
  P.bwd_rows = rows;
  off = 0;
  for (int i = 0; i < d->n_info_ops; ++i) { P.scr_info[i] = off; off += d->info_ops[i].in_dim * LD; }
  P.info_scratch_floats = off;
  auto add_fix = [&](const PmtLinearOp* ops, int n) {
    for (int i = 0; i < n; ++i)
      if (ops[i].flags & PMT_OP_SKIP_END) {
        SkipFix& f = P.skipfix[P.n_skipfix++];
        f.w_off = ops[i].w_off; f.b_off = ops[i].b_off; f.alpha_off = ops[i].alpha_off;
        f.n_w = ops[i].in_dim * ops[i].out_dim; f.n_b = ops[i].out_dim;
      }
  };
  add_fix(d->read_ops, d->n_read_ops); add_fix(d->info_ops, d->n_info_ops); add_fix(d->red_ops, d->n_red_ops);
  return 0;
}

int pmt_cnn_geometry(const Plan& P, CnnGeom* out) {
  CnnGeom& G = *out;
  memset(&G, 0, sizeof(G));
  const PmtModelDesc& d = P.d;
  int n_sp = 0;
  while (n_sp < d.n_cnn_ops && d.cnn_ops[n_sp].kind != PMT_CNN_LINEAR) ++n_sp;
  PMT_CHECK(n_sp < d.n_cnn_ops, "haplotype CNN must end with flatten + linear");
  for (int i = n_sp; i < d.n_cnn_ops; ++i) {
    PMT_CHECK(d.cnn_ops[i].kind == PMT_CNN_LINEAR, "spatial layer after flatten");
    PMT_CHECK(d.cnn_ops[i].out_ch <= 256 && (i == n_sp || d.cnn_ops[i].in_ch <= 256), "CNN linear layer too wide");
  }
  G.n_spatial = n_sp;
  int max_per_var = 10 * ((d.hap_len + 3) & ~3);
  G.lp[0] = (d.hap_len + 3) & ~3;
  int img = 0;
  for (int i = 0; i < n_sp; ++i) {
    const PmtCnnOp& op = d.cnn_ops[i];
    PMT_CHECK(op.ksize >= 1 && op.ksize <= 9, "conv/pool kernel_size %d unsupported (1..9)", op.ksize);
    G.lp[i + 1] = (op.out_len + 3) & ~3;
    const int ch = op.kind == PMT_CNN_CONV ? op.out_ch : op.in_ch;
    PMT_CHECK(ch <= 64 && op.in_ch <= 64, "CNN channels > 64 unsupported");
    if (ch * G.lp[i + 1] > max_per_var) max_per_var = ch * G.lp[i + 1];
    if (op.kind == PMT_CNN_CONV) {
      PMT_CHECK(op.stride == 1, "conv stride != 1 unsupported");
      G.img_off[i] = img;
      img += op.in_ch * op.ksize * ((op.out_ch + 7) / 8) * GROUP_STRIDE;
    }
  }
  G.img_total = (img + 3) & ~3;
  int imgT = 0;
  for (int i = 0; i < n_sp; ++i) {
    const PmtCnnOp& op = d.cnn_ops[i];
    if (op.kind != PMT_CNN_CONV) continue;
    G.imgT_off[i] = imgT;
    imgT += op.out_ch * op.ksize * ((op.in_ch + 7) / 8) * GROUP_STRIDE;
  }
  G.imgT_total = (imgT + 3) & ~3;
  // shared memory budget: 2 activation buffers + conv images + linear scratch
  const int budget_floats = (200 * 1024) / 4 - G.img_total;
  int vt = 32;
  for (; vt >= 1; --vt) {
    const int buf = 64 * 8 + vt * max_per_var + 64;  // + per-channel slack of 8 floats
    if (2 * buf + 2 * vt * 256 <= budget_floats) break;
  }
  PMT_CHECK(vt >= 1, "haplotype CNN does not fit in shared memory");
  G.vt = vt;
  G.buf_floats = ((64 * 8 + vt * max_per_var + 64) + 3) & ~3;
  return 0;
}

size_t pmt_image_bytes(const Plan& P, const CnnGeom& G) {
  return (size_t)(P.img_total + G.img_total + G.imgT_total + 64) * sizeof(float);
}

int pmt_sm_count() {
  int dev = 0, n_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n_sm < 1)
    return 148;   // no device: a B200's
  return n_sm;
}

// Test and measurement overrides of the call plan's choices, unset in normal use.  read_overrides is their only reader and
// pmt_call_plan its only caller, so every C-ABI call of the model, the size queries included, sees the same choices.
//   PMT_CNN_SINGLE=1       inference runs hap_cnn_tc_kernel over every layer; =0: the head + tail pair at any batch size
//   PMT_TC_PACKED=0        the sequential tile planner for every batch
//   PMT_LONG_SIMT=1        sets longer than a tile take the FP32 long-set kernel
//   PMT_BWD_CHUNK_TILES=n  the tensor-core backward recomputes and differentiates at most n >= 1 tiles per pass
struct Overrides {
  int cnn_single, tc_packed, long_simt, bwd_chunk_tiles;
};
static Overrides read_overrides() {
  auto get = [](const char* name) { const char* e = getenv(name); return e ? atoi(e) : -1; };
  return {get("PMT_CNN_SINGLE"), get("PMT_TC_PACKED"), get("PMT_LONG_SIMT"), get("PMT_BWD_CHUNK_TILES")};
}

// The posterior fit passes take no call plan; their override is read here, by its only reader:
//   PMT_POSTERIOR_CTAS=n   every problem of pmt_posterior_fit_pass / _many runs on a cluster of n CTAs (n = 1: the one-SM pass)
// -1 when unset, 0 when set to anything but 1, 2, 4, 8 or 16 (the callers refuse that).
int pmt_posterior_ctas_override() {
  const char* e = getenv("PMT_POSTERIOR_CTAS");
  if (!e) return -1;
  char* end = nullptr;
  const long n = strtol(e, &end, 10);
  return end != e && *end == '\0' && (n == 1 || n == 2 || n == 4 || n == 8 || n == 16) ? (int)n : 0;
}

// Batches below this size keep the sequential planner: packing saves ~5.5 % of the read kernel (1.13 ns per read), the packed
// planner costs ~0.1 ms more than the sequential one (one lane per claim places 512 sets), so it pays from ~2 M reads.
static const long long kPackedPlannerMinRows = 2000000;

static size_t info_kernel_smem(const Plan& P, InfoKernel k, int w4) {
  const PmtModelDesc& d = P.d;
  if (k == InfoKernel::TILE) {
    const int in_rows = d.n_info_features > PMT_MAX_DIM ? PMT_MAX_INFO_DIM : PMT_MAX_DIM;
    return (size_t)((in_rows + 2 * PMT_MAX_DIM) * LD + 2 * P.info_stage_floats) * sizeof(float);
  }
  size_t floats = 0;
  const int W = k == InfoKernel::WARP ? 32 : 4 * w4;
  if (k == InfoKernel::ROWS) {
    // the input tile: feature-major floats, or (raw16) a tile's fp16 rows as one span of up to 127 strides of I + 8 halves
    // plus a last row, which is the larger of the two below 8 features
    const size_t I = (size_t)d.n_info_features;
    const size_t raw16_words = ((INFO_TPB - 1) * (I + 8) + I + 1) / 2;
    floats = I * (INFO_TPB + 1) > raw16_words ? I * (INFO_TPB + 1) : raw16_words;
  }
  for (int i = 0; i < d.n_info_ops; ++i) floats += (size_t)(d.info_ops[i].in_dim + 1) * W;
  return floats * sizeof(float) + 16;
}

// reads_forward_kernel: aim for ~8 tiles per claim, but keep at least ~2 claims per SM when the batch is small
static Claims forward_claims(const PmtBatch* batch, int n_sm) {
  const double avg = (batch->n_variants > 0 && batch->n_rows > 0) ? (double)batch->n_rows / batch->n_variants : 16.0;
  Claims K;
  K.claim = (int)(8.0 * TILE / (avg + 1.0));
  const int by_parallelism = batch->n_variants / (2 * n_sm);
  if (K.claim > by_parallelism) K.claim = by_parallelism;
  if (K.claim > 512) K.claim = 512;
  if (K.claim < 1) K.claim = 1;
  K.n_claims = (batch->n_variants + K.claim - 1) / K.claim;
  K.grid = K.n_claims < n_sm ? K.n_claims : n_sm;
  return K;
}

int pmt_call_plan(const PmtModelDesc* desc, const PmtBatch* batch, bool train, CallPlan* out) {
  CallPlan& C = *out;
  memset(&C, 0, sizeof(C));
  if (pmt_build_plan(desc, &C.P) || pmt_cnn_geometry(C.P, &C.G)) return 1;
  const Plan& P = C.P;
  const Overrides ov = read_overrides();
  C.mode = pmt_precision_mode();
  C.passes = C.mode == PMT_PRECISION_TF32 ? 1 : 3;
  C.n_sm = pmt_sm_count();
  C.reads_tc_ok = pmt_tc_supported(P);
  pmt_tc_plan(P, &C.T);
  C.cnn_tc_ok = pmt_build_cnn_tc_plan(P, &C.C);
  C.cnn_bwd_ok = C.cnn_tc_ok && pmt_build_cnn_bwd_plan(P, C.C, &C.CB);
  C.cnn_split = C.cnn_tc_ok && pmt_build_cnn_split_plan(C.C, P.d.hap_len, &C.CH, &C.CT);
  const bool fp32 = C.mode == PMT_PRECISION_FP32;
  // the backward: the tensor-core read-path and haplotype-CNN kernels (pmt_tc_bwd.cu, pmt_cnn_bwd.cu) unless the FP32 mode
  // is selected or the model is outside their envelope, the FP32 SIMT kernels otherwise
  C.bwd_reads_tc = !fp32 && C.reads_tc_ok;
  C.bwd_cnn_tc = !fp32 && C.cnn_bwd_ok;
  C.saved = pmt_saved_layout(C, batch);
  train = train && C.saved.total > 0;
  const int B = batch ? batch->n_variants : 0;
  C.info_w4 = info_rows_w4(P.d);
  C.info = C.info_w4 == 0 ? InfoKernel::TILE : B <= 4096 ? InfoKernel::WARP : InfoKernel::ROWS;   // small batch: latency, not throughput
  C.info_smem = info_kernel_smem(P, C.info, C.info_w4);
  // the head + tail pair once the head kernel has a group for every SM; below that a call is a chain of latencies, and the
  // pair's second launch and global round trip cost more than the tail's MMA round trips it saves
  C.cnn = train                                        ? CnnKernel::TC_SAVE
          : fp32 || !C.cnn_tc_ok                        ? CnnKernel::SIMT
          : C.cnn_split && B >= (long long)C.CH.G * C.n_sm ? CnnKernel::TC_TAIL
                                                        : CnnKernel::TC;
  if (C.cnn == CnnKernel::TC || C.cnn == CnnKernel::TC_TAIL) {
    if (ov.cnn_single == 1) C.cnn = CnnKernel::TC;
    else if (ov.cnn_single == 0 && C.cnn_split) C.cnn = CnnKernel::TC_TAIL;
  }
  C.cnn_simt_smem = (size_t)(2 * C.G.buf_floats + C.G.img_total + 2 * C.G.vt * 256) * sizeof(float);
  C.reads = fp32 ? ReadsKernel::SIMT : train ? ReadsKernel::TC_SAVE : ReadsKernel::TC;
  C.packed_planner = C.reads == ReadsKernel::TC && batch && pmt_row_hint(batch) >= kPackedPlannerMinRows && ov.tc_packed != 0;
  C.ring = pmt_tc_ring(C.T, C.passes);
  C.ring_save = pmt_tc_ring(C.T, 3);
  C.reads_smem = tile_ctx_bytes(P, P.stage_floats);
  C.lng = !batch || !pmt_has_long_sets(batch)                                               ? LongKernel::NONE
          : !fp32 && ov.long_simt != 1 && pmt_tc_long_layout(P, batch, C.n_sm, &C.long_tc) ? LongKernel::TC
                                                                                          : LongKernel::SIMT;
  if (batch) {
    C.fwd_claims = forward_claims(batch, C.n_sm);
    const int n_sm = C.n_sm < PMT_PARTIAL_CTAS ? C.n_sm : PMT_PARTIAL_CTAS;
    C.fwd_long_grid = batch->n_variants < n_sm ? batch->n_variants : n_sm;
  }
  // who reads the SIMT images in a tensor-core mode: the tile-GEMM info MLP (widths outside info_mlp_rows_kernel), the SIMT
  // haplotype CNN (shapes outside the tensor-core envelope) -- and, depending on the batch, the FP32 long-set kernel
  C.simt_gemm = fp32 || C.info == InfoKernel::TILE;
  C.simt_conv = C.cnn == CnnKernel::SIMT;
  C.tc_bwd = pmt_tc_bwd_layout(C.T, batch, ov.bwd_chunk_tiles);
  C.ring_bwd = pmt_tc_bwd_ring(C.T);

  // refusals, in the order the kernels would run
  const bool info_fits = C.info == InfoKernel::TILE || C.info_smem <= 200 * 1024;
  const bool ring_fits = (C.reads != ReadsKernel::TC_SAVE || C.ring_save.n_stages >= 2) &&
                         ((C.reads != ReadsKernel::TC && C.lng != LongKernel::TC) || C.ring.n_stages >= 2);
  const char* fwd_why = !info_fits                                       ? "info MLP does not fit in shared memory"
                        : C.reads != ReadsKernel::SIMT && !C.reads_tc_ok ? "this model shape is outside the tensor-core kernel's envelope; use PMT_PRECISION_FP32"
                        : !ring_fits                                     ? "tensor-core forward: weight ring does not fit in shared memory"
                                                                         : "";
  snprintf(C.fwd_refusal, sizeof(C.fwd_refusal), "%s", fwd_why);
  // the backward recomputes the info MLP when the forward's embeddings are not passed in, and the read path's forward
  // operands when they were not saved
  pmt_plan_backward(C, batch);
  if (!C.bwd_refusal[0]) {
    const char* bwd_why = !info_fits                                          ? "info MLP does not fit in shared memory"
                          : C.bwd_reads_tc && C.ring_save.n_stages < 2        ? "tensor-core forward: weight ring does not fit in shared memory"
                          : C.bwd_reads_tc && C.ring_bwd.n_stages < 2         ? "tensor-core backward: weight ring does not fit in shared memory"
                                                                              : "";
    snprintf(C.bwd_refusal, sizeof(C.bwd_refusal), "%s", bwd_why);
  }
  pmt_plan_workspaces(C, batch);
  return 0;
}

int pmt_launch_prepare(const CallPlan& C, const float* weights, float* image, cudaStream_t st, bool gemm, bool conv) {
  const Plan& P = C.P;
  const CnnGeom& G = C.G;
  if (gemm) pack_weights_kernel<<<dim3(P.n_gemm, 4), 256, 0, st>>>(P, weights, image);
  if (conv && G.n_spatial > 0) pack_conv_kernel<<<G.n_spatial, 256, 0, st>>>(P, G, weights, image + P.img_total);
  if (conv && G.n_spatial > 0) pack_convT_kernel<<<G.n_spatial, 256, 0, st>>>(P, G, weights, image + P.img_total);
  return 0;
}

int pmt_launch_info_mlp(const CallPlan& C, const float* weights, const float* image, const PmtBatch* batch, float* info_seq,
                        cudaStream_t st) {
  const Plan& P = C.P;
  const int B = batch->n_variants;
  const size_t smem = C.info_smem;
  if (C.info == InfoKernel::WARP) {
    PMT_CUDA(cudaFuncSetAttribute(info_mlp_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int blocks = (B + INFO_WARPS - 1) / INFO_WARPS;
    info_mlp_warp_kernel<<<blocks < 148 * 4 ? blocks : 148 * 4, 32 * INFO_WARPS, smem, st>>>(P.d, weights, batch->info, batch->info_kind,
                                                                                               batch->info_stride, B, info_seq);
  } else if (C.info == InfoKernel::ROWS) {
    switch (C.info_w4) {
      case 1: return launch_info_rows<1>(P.d, weights, batch, info_seq, smem, st);
      case 2: return launch_info_rows<2>(P.d, weights, batch, info_seq, smem, st);
      case 3: return launch_info_rows<3>(P.d, weights, batch, info_seq, smem, st);
      case 4: return launch_info_rows<4>(P.d, weights, batch, info_seq, smem, st);
      case 5: return launch_info_rows<5>(P.d, weights, batch, info_seq, smem, st);
      case 6: return launch_info_rows<6>(P.d, weights, batch, info_seq, smem, st);
      case 7: return launch_info_rows<7>(P.d, weights, batch, info_seq, smem, st);
      default: return launch_info_rows<8>(P.d, weights, batch, info_seq, smem, st);
    }
  } else {
    PMT_CUDA(cudaFuncSetAttribute(info_mlp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    info_mlp_kernel<<<(B + TILE - 1) / TILE, NTHREADS, smem, st>>>(P, weights, image, batch->info, batch->info_kind,
                                                                   batch->info_stride, B, info_seq);
  }
  return 0;
}

int pmt_launch_hap_cnn_simt(const CallPlan& C, const float* weights, const float* image, const PmtBatch* batch, float* info_seq,
                            cudaStream_t st) {
  const CnnGeom& G = C.G;
  const int B = batch->n_variants;
  PMT_CUDA(cudaFuncSetAttribute(hap_cnn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C.cnn_simt_smem));
  int grid = (B + G.vt - 1) / G.vt;
  if (grid > 148 * 4) grid = 148 * 4;
  hap_cnn_kernel<<<grid, NTHREADS, C.cnn_simt_smem, st>>>(C.P, G, weights, image + C.P.img_total, batch->haplotypes, batch->hap_kind,
                                               batch->hap_stride, B, info_seq);
  return 0;
}

static int forward_impl(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                        void* workspace, size_t workspace_bytes, void* stream, bool reuse_images, unsigned char* saved = nullptr,
                        size_t saved_bytes = 0) {
  CallPlan C;
  if (pmt_call_plan(desc, batch, saved != nullptr, &C)) return 1;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  FwdBuffers W;
  if (pmt_forward_buffers(C, workspace, workspace_bytes, &W)) return 1;
  PMT_CHECK(batch->n_variants > 0, "empty batch");
  PMT_CHECK(!C.fwd_refusal[0], "%s", C.fwd_refusal);
  SavedBuffers S{};
  if (saved) {
    PMT_CHECK(C.saved.total > 0 && saved_bytes >= C.saved.total,
              "pmt_forward_train: no saved-forward path for this call or buffer too small (%zu < %zu)", saved_bytes, C.saved.total);
    PMT_CHECK((reinterpret_cast<uintptr_t>(saved) & 255) == 0, "pmt_forward_train: the saved buffer must be 256-byte aligned");
    if (pmt_saved_buffers(C, saved, saved_bytes, &S)) return 1;
  }
  float* image = W.image;
  float* info_seq = out->info_seq_be ? out->info_seq_be : W.info_seq;
  PMT_CUDA(cudaMemsetAsync(W.counters, 0, C.fwd.counters.bytes, st));
  {
    // a prepared call finds the images of the model; the FP32 long-set kernel's depend on the batch
    const bool simt_long = C.lng == LongKernel::SIMT;
    if (!reuse_images) pmt_launch_prepare(C, weights, image, st, C.simt_gemm || simt_long, C.simt_conv);
    else if (simt_long && !C.simt_gemm) pmt_launch_prepare(C, weights, image, st, true, false);
  }
  // per-variant embeddings: the info MLP, then the haplotype CNN (in training its SAVE variant: same results, activations kept)
  if (pmt_launch_info_mlp(C, weights, image, batch, info_seq, st)) return 1;
  switch (C.cnn) {
    case CnnKernel::TC:
    case CnnKernel::TC_TAIL:
      if (pmt_launch_cnn_tc(C, weights, batch, info_seq, W, reuse_images, st)) return 1;
      break;
    case CnnKernel::TC_SAVE:
      if (pmt_cnn_forward_train(C, weights, batch, info_seq, W.cnn_tc_image, S.cnn, st)) return 1;
      break;
    case CnnKernel::SIMT:
      if (pmt_launch_hap_cnn_simt(C, weights, image, batch, info_seq, st)) return 1;
      break;
  }

  Plan P = C.P;
  P.claim_variants = C.fwd_claims.claim;
  ReadKernelArgs A;
  A.wflat = weights; A.image = image; A.batch = *batch; A.out = *out; A.out.info_seq_be = info_seq; A.claim_counter = W.counters;
  A.scratch = nullptr; A.scratch_stride = 0;
  const size_t smem = C.reads_smem;
  PMT_CUDA(cudaFuncSetAttribute(reads_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  PmtOutputs o2 = *out;
  o2.info_seq_be = info_seq;
  if (C.reads == ReadsKernel::SIMT) {
    pmt_profile_begin(st);
    reads_forward_kernel<<<C.fwd_claims.grid, NTHREADS, smem, st>>>(P, A);
    pmt_profile_end(st);
  } else {
    if (C.reads == ReadsKernel::TC_SAVE) {   // deterministic tile list + the SAVE variant of the read kernel, operands kept for the backward
      if (pmt_tc_forward_train(C, weights, batch, &o2, W, S, st)) return 1;
    } else if (pmt_launch_reads_tc(C, weights, batch, &o2, W, reuse_images, st)) {
      return 1;
    }
  }
  if (C.lng == LongKernel::TC) {
    // sets longer than a tile, cut into single-side tiles on the same tensor-core pipeline (pmt_tc.cuh: LongTile)
    if (pmt_launch_reads_tc_long(C, weights, batch, &o2, W, st)) return 1;
  } else if (C.lng == LongKernel::SIMT) {
    A.scratch = W.long_scratch;
    A.scratch_stride = (long long)C.fwd.long_scratch_floats;
    PMT_CUDA(cudaFuncSetAttribute(reads_forward_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    reads_forward_long_kernel<<<C.fwd_long_grid, NTHREADS, smem, st>>>(P, A);
  }
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_forward launch failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int pmt_forward(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                           void* workspace, size_t workspace_bytes, void* stream) {
  return forward_impl(desc, weights, batch, out, workspace, workspace_bytes, stream, false);
}

extern "C" int pmt_forward_train(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                                 void* workspace, size_t workspace_bytes, void* saved, size_t saved_bytes, void* stream) {
  PMT_CHECK(saved != nullptr, "pmt_forward_train: saved buffer missing (pmt_train_saved_bytes() == 0 means: call pmt_forward)");
  return forward_impl(desc, weights, batch, out, workspace, workspace_bytes, stream, false, reinterpret_cast<unsigned char*>(saved), saved_bytes);
}

extern "C" int pmt_forward_prepared(const PmtModelDesc* desc, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  return forward_impl(desc, weights, batch, out, workspace, workspace_bytes, stream, true);
}

extern "C" int pmt_decode_reads(const uint8_t* reads_u8, int64_t n_rows, int32_t row_bytes, float* out, void* stream) {
  PMT_CHECK(row_bytes >= 7, "row_bytes %d < 7 packed bytes", row_bytes);
  if (n_rows == 0) return 0;
  const long long total = (long long)n_rows * (56 + row_bytes - 7);
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  decode_reads_kernel<<<(int)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(reads_u8, n_rows, row_bytes, out);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "pmt_decode_reads launch failed: %s", cudaGetErrorString(e));
  return 0;
}
