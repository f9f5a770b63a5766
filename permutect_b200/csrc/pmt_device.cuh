// Device-side building blocks shared by the forward and backward kernels (sm_100a).
//
// Data layout inside a CTA: a tile of up to TILE reads (rows) is held FEATURE-MAJOR in shared memory,
// buf[f * LD + r], so that (a) per-row work (LayerNorm, gating, decode) has lane == row and is
// bank-conflict free, and (b) the register-tiled FP32 GEMM reads 4 consecutive rows of one feature
// as a single 16-byte LDS.  Weights of the GEMM being executed are staged in shared memory with
// cp.async, double-buffered, from packed images built once per call by pack_weights_kernel.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/permutect_b200.h"

namespace pmt {

constexpr int TILE = PMT_TILE_ROWS;  // rows (reads, or variants in the per-variant kernels) per CTA tile
constexpr int LD = TILE + 4;         // row stride of the feature-major activation buffers (floats)
constexpr int NTHREADS = 256;
constexpr int NWARPS = NTHREADS / 32;
constexpr int NPART = NTHREADS / TILE;   // threads per tile row; thread (row, part) = (tid % TILE, tid / TILE)
// Part `part` of a per-row loop over n items covers [part_lo(n, part), part_lo(n, part + 1)).
__device__ __forceinline__ int part_lo(int n, int part) { return (n * part) / NPART; }
constexpr int MAX_GEMM = 96;
constexpr int GROUP_STRIDE = 8;      // floats per column group in a packed weight image row

constexpr float SELU_ALPHA = 1.6732632423543772848170429916717f;
constexpr float SELU_SCALE = 1.0507009873554804934193349852946f;
constexpr float LN_EPS = 1e-5f;
constexpr float LOG_2PI = 1.8378770664093453f;

// One staged GEMM: Y[n][r] = sum_k W[n][k] X[k][r] + b[n].  The packed image is [K][G][8] floats
// (column n lives at group n / NT, slot n % NT; unused slots are zero).  `dual` ops carry a second
// image/bias for alt rows (proj1/proj2 of the gated block, gated_mlp.py:165-171).
// The TRANSPOSED image of the same op (imgT_*, GT, NTT) serves the backward data-gradient GEMM
// dX[k][r] = sum_n W[n][k] dY[n][r]: reduction length N, K outputs.
struct GemmOp {
  int K, N, G, NT;
  int img_off;     // float offset of the (ref) image inside the packed buffer; alt image follows it
  int img_floats;  // floats staged for this op (both images when dual)
  int w_off, b_off, w_alt_off, b_alt_off;  // flat-weight offsets; *_alt_off < 0 when not dual
  int GT, NTT, imgT_off, imgT_floats;
};

struct SkipFix {   // DenseSkipBlock last layer: backward accumulates the un-scaled U = dx_out . s^T (see reduce kernel)
  int w_off, b_off, alpha_off, n_w, n_b;
};

struct Plan {
  PmtModelDesc d;
  int n_gemm;
  int read_g0, info_g0, red_g0, blk_g0;  // first GemmOp of each program; block b uses blk_g0 + 2b (+1)
  int img_total;                         // floats in the packed image buffer (forward + transposed images)
  int stage_floats;                      // largest staged image of the read-path ops (forward and transposed)
  int info_stage_floats;
  int sum_w;                             // width of the per-variant sum scratch: max(d_ffn/2, d_feat)
  int claim_variants;                    // variants claimed per scheduling step
  // per-CTA activation scratch of the backward kernel: feature-major [nf][LD] images, float offsets
  int scr_read[PMT_MAX_MLP_OPS + 1];     // input of read op i
  int scr_red[PMT_MAX_MLP_OPS + 1];      // input of reducer op i; [n_red_ops] = reducer output y
  int scr_x[PMT_MAX_BLOCKS];             // x entering gated block b
  int scr_z[PMT_MAX_BLOCKS];             // z = SELU(proj1(LN x)) of block b (before the SGU LayerNorm)
  int scr_info[PMT_MAX_MLP_OPS + 1];     // input of info op i (info MLP backward kernel)
  int scratch_floats, info_scratch_floats;
  int bwd_rows;                          // feature rows per backward activation buffer
  int n_skipfix;
  SkipFix skipfix[3 * PMT_MAX_MLP_OPS];
  GemmOp gemm[MAX_GEMM];
};

struct CnnGeom {
  int vt;                        // variants per CTA pass
  int lp[PMT_MAX_CNN_OPS + 1];   // padded per-variant length of the activation entering op i (lp[n] = after last)
  int img_off[PMT_MAX_CNN_OPS];  // conv image offsets (floats) inside the conv image buffer
  int img_total;
  int imgT_off[PMT_MAX_CNN_OPS]; // flipped + transposed conv images (backward data gradient), after the forward ones
  int imgT_total;
  int buf_floats;                // floats per ping-pong activation buffer
  int n_spatial;                 // ops before the first PMT_CNN_LINEAR
};

// Branch-free: the exponential is evaluated for every lane (argument clamped to <= 0) and selected.
__device__ __forceinline__ float selu(float x) {
  const float neg = SELU_ALPHA * (expf(fminf(x, 0.f)) - 1.f);
  return SELU_SCALE * (x > 0.f ? x : neg);
}
// d selu / dx expressed through the OUTPUT y = selu(x): y > 0 -> scale, else y + scale*alpha
__device__ __forceinline__ float selu_grad_from_out(float y) {
  return y > 0.f ? SELU_SCALE : y + SELU_SCALE * SELU_ALPHA;
}
__device__ __forceinline__ float sigmoidf(float x) { return 1.f / (1.f + expf(-x)); }   // torch.sigmoid
__device__ __forceinline__ unsigned smem_addr(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ float4 lds128(unsigned a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(unsigned a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
// cp.async of 16 bytes of which the first src_bytes come from global memory (the rest is zero-filled)
__device__ __forceinline__ void cp_async16_zfill(void* smem, const void* gmem, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(smem_addr(smem)), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// fp32 -> TF32 rounded to nearest: the operand precision of the TF32 tensor-core instructions
__device__ __forceinline__ float rna_tf32(float v) {
  unsigned r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
// c += a b: one warp-level m16n8k8 TF32 MMA (mma.sync), fp32 accumulators
__device__ __forceinline__ void mma_tf32(float* c, const float* a, float b0, float b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(__float_as_uint(a[0])), "r"(__float_as_uint(a[1])), "r"(__float_as_uint(a[2])), "r"(__float_as_uint(a[3])),
                 "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}

// Double-buffered weight stage.  All control flow is CTA-uniform.  Keys: g for the forward image of
// GemmOp g, MAX_GEMM + g for its transposed image.
struct Stage {
  float* buf0;
  float* buf1;
  int res0, res1;   // key held (or in flight) in each buffer, -1 = none
  int last;         // buffer most recently acquired
  bool pending;     // a prefetch into the other buffer has been issued and not yet acquired
  const float* image;
  const Plan* plan;

  __device__ __forceinline__ void init(float* b0, float* b1, const float* img, const Plan* p) {
    buf0 = b0; buf1 = b1; res0 = res1 = -1; last = 1; pending = false; image = img; plan = p;
  }
  __device__ __forceinline__ void issue(int slot, int key) {
    const bool tr = key >= MAX_GEMM;
    const GemmOp& op = plan->gemm[tr ? key - MAX_GEMM : key];
    const float4* src = reinterpret_cast<const float4*>(image + (tr ? op.imgT_off : op.img_off));
    const int n4 = (tr ? op.imgT_floats : op.img_floats) / 4;
    float4* dst = reinterpret_cast<float4*>(slot ? buf1 : buf0);
    for (int i = threadIdx.x; i < n4; i += NTHREADS) cp_async16(dst + i, src + i);
    cp_async_commit();
    if (slot) res1 = key; else res0 = key;
  }
  // Start loading `key` (if it is not already resident) into the buffer that is NOT in use.
  __device__ __forceinline__ void prefetch(int key) {
    if (key < 0 || pending || res0 == key || res1 == key) return;
    issue(last ^ 1, key);
    pending = true;
  }
  // Make `key` available; contains a __syncthreads() (which also orders the preceding activation writes).
  __device__ __forceinline__ const float* acquire(int key) {
    int slot = res0 == key ? 0 : (res1 == key ? 1 : -1);
    if (slot < 0) {
      slot = last ^ 1;
      cp_async_wait_all();
      __syncthreads();  // nobody still reads buf[slot], no copy into it is in flight
      issue(slot, key);
    }
    cp_async_wait_all();
    __syncthreads();
    last = slot;
    pending = false;
    return slot ? buf1 : buf0;
  }
};

// Epilogue: Y = (ACC ? Y : 0) + alpha * (SELU ? selu(v) : v) * (DSELU ? selu'(act) : 1)
enum EpilogueFlags { EPI_STORE = 0, EPI_SELU = 1, EPI_ACC = 2, EPI_DSELU = 4 };
constexpr int EPI_RESIDUAL = EPI_ACC;

template <int NT>
__device__ __noinline__ void gemm_tile_nt(unsigned x_s, int K, int N, int G, bool dual, int b_off, int b_alt_off,
                                          unsigned img_s, const float* __restrict__ wflat, int ref_rows_padded,
                                          unsigned y_s, int flags, float alpha, unsigned act_s, int rows_used) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = lane * 4;
  if (r0 >= rows_used) return;
  const bool is_alt = dual && (r0 >= ref_rows_padded);
  const int wstride = G * GROUP_STRIDE * 4;  // bytes
  const unsigned wimg = img_s + (is_alt ? K * wstride : 0);
  const int boff = is_alt ? b_alt_off : b_off;
  for (int g = warp; g < G; g += NWARPS) {
    float acc[4][NT];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const int n = g * NT + j;
      const float b = (boff >= 0 && n < N) ? __ldg(wflat + boff + n) : 0.f;
      acc[0][j] = b; acc[1][j] = b; acc[2][j] = b; acc[3][j] = b;
    }
    unsigned xp = x_s + r0 * 4;
    unsigned wp = wimg + g * GROUP_STRIDE * 4;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
      const float4 x = lds128(xp);
      float w[8];
      const float4 w0 = lds128(wp);
      w[0] = w0.x; w[1] = w0.y; w[2] = w0.z; w[3] = w0.w;
      if (NT > 4) {
        const float4 w1 = lds128(wp + 16);
        w[4] = w1.x; w[5] = w1.y; w[6] = w1.z; w[7] = w1.w;
      }
      xp += LD * 4;
      wp += wstride;
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        acc[0][j] = fmaf(x.x, w[j], acc[0][j]);
        acc[1][j] = fmaf(x.y, w[j], acc[1][j]);
        acc[2][j] = fmaf(x.z, w[j], acc[2][j]);
        acc[3][j] = fmaf(x.w, w[j], acc[3][j]);
      }
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const int n = g * NT + j;
      if (n < N) {
        const unsigned off = (n * LD + r0) * 4;
        float4 v = make_float4(acc[0][j], acc[1][j], acc[2][j], acc[3][j]);
        if (flags & EPI_SELU) { v.x = selu(v.x); v.y = selu(v.y); v.z = selu(v.z); v.w = selu(v.w); }
        if (flags & EPI_DSELU) {
          const float4 a = lds128(act_s + off);
          v.x *= selu_grad_from_out(a.x); v.y *= selu_grad_from_out(a.y);
          v.z *= selu_grad_from_out(a.z); v.w *= selu_grad_from_out(a.w);
        }
        if (flags & EPI_ACC) {
          const float4 o = lds128(y_s + off);
          v.x = fmaf(alpha, v.x, o.x); v.y = fmaf(alpha, v.y, o.y); v.z = fmaf(alpha, v.z, o.z); v.w = fmaf(alpha, v.w, o.w);
        } else if (alpha != 1.f) {
          v.x *= alpha; v.y *= alpha; v.z *= alpha; v.w *= alpha;
        }
        sts128(y_s + off, v);
      }
    }
  }
}

#define PMT_GEMM_DISPATCH(NTV, ...)                        \
  switch (NTV) {                                           \
    case 1: gemm_tile_nt<1>(__VA_ARGS__); break;           \
    case 2: gemm_tile_nt<2>(__VA_ARGS__); break;           \
    case 3: gemm_tile_nt<3>(__VA_ARGS__); break;           \
    case 4: gemm_tile_nt<4>(__VA_ARGS__); break;           \
    case 5: gemm_tile_nt<5>(__VA_ARGS__); break;           \
    case 6: gemm_tile_nt<6>(__VA_ARGS__); break;           \
    case 7: gemm_tile_nt<7>(__VA_ARGS__); break;           \
    default: gemm_tile_nt<8>(__VA_ARGS__); break;          \
  }

// Y <- epilogue(W X + b) over the tile (forward).  X and Y must be different buffers unless the
// epilogue accumulates into a Y disjoint from X.  Caller synchronises before consumers read Y.
__device__ __forceinline__ void gemm_tile(const float* X, const GemmOp& op, const float* img, const float* wflat,
                                          int ref_rows_padded, float* Y, int flags, float alpha, int rows_used) {
  const unsigned xs = smem_addr(X), is = smem_addr(img), ys = smem_addr(Y);
  PMT_GEMM_DISPATCH(op.NT, xs, op.K, op.N, op.G, op.w_alt_off >= 0, op.b_off, op.b_alt_off, is, wflat,
                    ref_rows_padded, ys, flags, alpha, 0u, rows_used)
}

// dX <- epilogue(W^T dY) over the tile (backward data gradient), using the transposed image.
__device__ __forceinline__ void gemm_tile_T(const float* dY, const GemmOp& op, const float* imgT, int ref_rows_padded,
                                            float* dX, int flags, float alpha, const float* act, int rows_used) {
  const unsigned xs = smem_addr(dY), is = smem_addr(imgT), ys = smem_addr(dX);
  const unsigned as = act ? smem_addr(act) : 0u;
  PMT_GEMM_DISPATCH(op.NTT, xs, op.N, op.K, op.GT, op.w_alt_off >= 0, -1, -1, is, nullptr, ref_rows_padded, ys, flags,
                    alpha, as, rows_used)
}

// Fire-and-forget accumulation into a CTA-private gradient buffer: a reduction does not wait for the old value the way
// a load-add-store does.  Every address is only ever updated by one thread of one CTA, in program order, so the result
// is still bitwise reproducible.
__device__ __forceinline__ void red_add(float* p, float v) { asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }

// Weight gradient: part[n*K + k] += sum_{r in [r_lo, r_hi)} dY[n][r] * A[k][r]   (r_lo, r_hi multiples of 4).
// `part` is this CTA's private gradient buffer, so the read-modify-write needs no atomics and the
// summation order is fixed.  Lanes 0-15 / 16-31 of a warp take two groups of 4 consecutive n; each
// lane takes k in {kl, kl+16, kl+32, kl+48}: 16 consecutive feature rows per LDS -> conflict-free.
// (Giving a warp one n-group and 32 lanes along k when N <= 4 NWARPS was measured: no gain.)
// One (4 n) x (KA k per lane) unit of wgrad_tile; KA is a template parameter so that no issue slot goes to
// predicated-off FMAs (a runtime bound on a 4 x 4 unit wasted half of them at K = 30 and three quarters at K = 10).
template <int KA>
__device__ __forceinline__ void wgrad_unit(unsigned dy_s, int N, unsigned a_s, int K, float* __restrict__ part, int r_lo,
                                           int r_hi, int ng, int k_first, int k_step) {
  float acc[4][KA];
#pragma unroll
  for (int b = 0; b < 4; ++b)
#pragma unroll
    for (int a = 0; a < KA; ++a) acc[b][a] = 0.f;
  unsigned dyp[4], ap[KA];
#pragma unroll
  for (int b = 0; b < 4; ++b) dyp[b] = dy_s + (min(ng * 4 + b, N - 1) * LD) * 4;
#pragma unroll
  for (int a = 0; a < KA; ++a) ap[a] = a_s + (min(k_first + k_step * a, K - 1) * LD) * 4;
  for (int r = r_lo; r < r_hi; r += 4) {
    float4 dy[4], av[KA];
#pragma unroll
    for (int b = 0; b < 4; ++b) dy[b] = lds128(dyp[b] + r * 4);
#pragma unroll
    for (int a = 0; a < KA; ++a) av[a] = lds128(ap[a] + r * 4);
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int a = 0; a < KA; ++a) {
        acc[b][a] = fmaf(dy[b].x, av[a].x, acc[b][a]);
        acc[b][a] = fmaf(dy[b].y, av[a].y, acc[b][a]);
        acc[b][a] = fmaf(dy[b].z, av[a].z, acc[b][a]);
        acc[b][a] = fmaf(dy[b].w, av[a].w, acc[b][a]);
      }
  }
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    const int n = ng * 4 + b;
    if (n < N) {
#pragma unroll
      for (int a = 0; a < KA; ++a) {
        const int k = k_first + k_step * a;
        if (k < K) red_add(part + n * K + k, acc[b][a]);
      }
    }
  }
}

static __device__ __noinline__ void wgrad_tile(unsigned dy_s, int N, unsigned a_s, int K, float* __restrict__ part,
                                               int r_lo, int r_hi) {
  if (r_hi <= r_lo) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kl = lane & 15;
  for (int k0 = 0; k0 < K; k0 += 64) {
    const int ka = min(4, (K - k0 + 15) >> 4);
    for (int ng = warp * 2 + (lane >> 4); ng * 4 < N; ng += 2 * NWARPS) {
      switch (ka) {
        case 1: wgrad_unit<1>(dy_s, N, a_s, K, part, r_lo, r_hi, ng, k0 + kl, 16); break;
        case 2: wgrad_unit<2>(dy_s, N, a_s, K, part, r_lo, r_hi, ng, k0 + kl, 16); break;
        case 3: wgrad_unit<3>(dy_s, N, a_s, K, part, r_lo, r_hi, ng, k0 + kl, 16); break;
        default: wgrad_unit<4>(dy_s, N, a_s, K, part, r_lo, r_hi, ng, k0 + kl, 16); break;
      }
    }
  }
}

// part[f * stride] += sum_{r in [r_lo, r_hi)} buf[f][r] * (other ? other[f][r] : 1)  for f < nf.  A warp reduces four
// features at a time (four independent shuffle trees in flight; one tree per iteration left the warp waiting on
// shuffle latency: 1.7 k cycles per 30 features).
__device__ __forceinline__ void rowdot_tile(const float* buf, const float* other, int nf, float* __restrict__ part,
                                            int r_lo, int r_hi, int stride = 1) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = r_lo + lane * 4;
  for (int f0 = warp * 4; f0 < nf; f0 += NWARPS * 4) {
    float s[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int f = f0 + q;
      s[q] = 0.f;
      if (f < nf && r < r_hi) {
        const float4 v = *reinterpret_cast<const float4*>(buf + f * LD + r);
        if (other) {
          const float4 o = *reinterpret_cast<const float4*>(other + f * LD + r);
          s[q] = v.x * o.x + v.y * o.y + v.z * o.z + v.w * o.w;
        } else {
          s[q] = v.x + v.y + v.z + v.w;
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int q = 0; q < 4; ++q) s[q] += __shfl_xor_sync(0xffffffffu, s[q], o);
    const float mine = lane == 0 ? s[0] : (lane == 1 ? s[1] : (lane == 2 ? s[2] : s[3]));
    if (lane < 4 && f0 + lane < nf) red_add(part + (f0 + lane) * stride, mine);
  }
}

// Deterministic CTA-wide sum of per-thread contributions to up to `cap` scalars.  Every thread calls
// add(i, v) for each scalar i (warp-uniform i), then after a __syncthreads() flush() adds the totals
// into part[] in a fixed order.
struct BlockAccum {
  float* wpart;   // shared [NWARPS][cap]
  int cap;
  __device__ __forceinline__ void init(float* smem_buf, int capacity) { wpart = smem_buf; cap = capacity; }
  __device__ __forceinline__ void add(int i, float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) wpart[(threadIdx.x >> 5) * cap + i] = v;
  }
  // dst[i] += total of scalar (first + i) for i < n   (call after a __syncthreads())
  __device__ __forceinline__ void flush(float* __restrict__ dst, int first, int n) {
    for (int i = threadIdx.x; i < n; i += NTHREADS) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < NWARPS; ++w) s += wpart[w * cap + first + i];
      dst[i] += s;
    }
  }
};

// dst[f][r] = selu(src[f][r]) for f < nf (all TILE rows; padding rows hold finite garbage)
__device__ __forceinline__ void selu_copy(const float* src, float* dst, int nf) {
  for (int i = threadIdx.x; i < nf * (TILE / 4); i += NTHREADS) {
    const int f = i / (TILE / 4), q = i % (TILE / 4);
    float4 v = *reinterpret_cast<const float4*>(src + f * LD + q * 4);
    v.x = selu(v.x); v.y = selu(v.y); v.z = selu(v.z); v.w = selu(v.w);
    *reinterpret_cast<float4*>(dst + f * LD + q * 4) = v;
  }
}
__device__ __forceinline__ void copy_features(const float* src, float* dst, int nf) {
  for (int i = threadIdx.x; i < nf * (TILE / 4); i += NTHREADS) {
    const int f = i / (TILE / 4), q = i % (TILE / 4);
    *reinterpret_cast<float4*>(dst + f * LD + q * 4) = *reinterpret_cast<const float4*>(src + f * LD + q * 4);
  }
}
// dst[f][r] *= selu'(act[f][r])
__device__ __forceinline__ void mul_dselu(float* dst, const float* act, int nf) {
  for (int i = threadIdx.x; i < nf * (TILE / 4); i += NTHREADS) {
    const int f = i / (TILE / 4), q = i % (TILE / 4);
    float4 v = *reinterpret_cast<const float4*>(dst + f * LD + q * 4);
    const float4 a = *reinterpret_cast<const float4*>(act + f * LD + q * 4);
    v.x *= selu_grad_from_out(a.x); v.y *= selu_grad_from_out(a.y);
    v.z *= selu_grad_from_out(a.z); v.w *= selu_grad_from_out(a.w);
    *reinterpret_cast<float4*>(dst + f * LD + q * 4) = v;
  }
}

// feature-major image <-> global scratch (nf features, all LD columns; 16-byte vectors)
__device__ __forceinline__ void save_rows(const float* buf, int nf, float* g) {
  const float4* s4 = reinterpret_cast<const float4*>(buf);
  float4* g4 = reinterpret_cast<float4*>(g);
  for (int i = threadIdx.x; i < nf * (LD / 4); i += NTHREADS) g4[i] = s4[i];
}
// global -> shared with cp.async: every copy of the thread is in flight at once (a register round trip serialised one
// L2 / DRAM latency per 16 bytes: 4.5 k cycles per 30-feature image).  The thread waits for its own copies; the caller's
// __syncthreads() publishes them.
__device__ __forceinline__ void load_rows_async(float* buf, int nf, const float* g) {   // caller: cp_async_wait_all()
  float4* s4 = reinterpret_cast<float4*>(buf);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  for (int i = threadIdx.x; i < nf * (LD / 4); i += NTHREADS) cp_async16(s4 + i, g4 + i);
  cp_async_commit();
}
__device__ __forceinline__ void load_rows(float* buf, int nf, const float* g) {
  load_rows_async(buf, nf, g);
  cp_async_wait_all();
}

// Runs an MLP program (mlp.py:25-76) over the tile.  `cur` holds the input; b0/b1/b2 are the three
// activation buffers (cur is one of them).  Returns the buffer holding the output.
// next_after: stage key to prefetch while the last layer runs (-1 = none).
// scr != nullptr: the activation entering every op is saved to scr + scr_off[i] (backward recompute pass).
static __device__ __noinline__ float* run_mlp(const Plan& P, const PmtLinearOp* ops, int n_ops, int g0, float* cur,
                                              float* b0, float* b1, float* b2, Stage& stage, const float* wflat,
                                              int rows_used, int next_after, float* scr = nullptr,
                                              const int* scr_off = nullptr) {
  float* res = nullptr;
  for (int i = 0; i < n_ops; ++i) {
    const PmtLinearOp& lop = ops[i];
    const GemmOp& gop = P.gemm[g0 + i];
    float* src = cur;
    if (lop.flags & PMT_OP_SKIP_BEGIN) {
      res = cur;
      float* tmp = (b0 != cur) ? b0 : b1;
      __syncthreads();  // producers of `cur` are done
      if (scr) save_rows(cur, lop.in_dim, scr + scr_off[i]);
      selu_copy(cur, tmp, lop.in_dim);
      src = tmp;
    }
    const float* img = stage.acquire(g0 + i);
    stage.prefetch(i + 1 < n_ops ? g0 + i + 1 : next_after);
    if (scr && !(lop.flags & PMT_OP_SKIP_BEGIN)) save_rows(cur, lop.in_dim, scr + scr_off[i]);
    if (lop.flags & PMT_OP_SKIP_END) {
      gemm_tile(src, gop, img, wflat, 0, res, EPI_RESIDUAL, __ldg(wflat + lop.alpha_off), rows_used);
      cur = res;
      res = nullptr;
    } else {
      float* dst = b0;
      if (dst == src || dst == res) dst = b1;
      if (dst == src || dst == res) dst = b2;
      gemm_tile(src, gop, img, wflat, 0, dst, (lop.flags & PMT_OP_POST_SELU) ? EPI_SELU : EPI_STORE, 1.f, rows_used);
      cur = dst;
    }
  }
  return cur;
}

}  // namespace pmt
