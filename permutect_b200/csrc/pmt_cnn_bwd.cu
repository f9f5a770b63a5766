// Tensor-core backward of the haplotype CNN (autograd of dna_sequence_convolution.py:57-111 as driven by
// misc_utils.py:125-129) for sm_100a.
//
// The forward recompute is the tcgen05 kernel of pmt_cnn_tc.cu in its SAVE variant: it leaves every layer's activation a_l
// (and, where a max-pool of two is fused, which element of each window won) in global memory.  This kernel then walks the
// layers in reverse for groups of VT variants held in shared memory.  Per layer l:
//
//   dY_l   = route(g_l through the pool) * act'(a_l)              one (channel, variant) row per warp trip, zero margins
//   dW_l  += dY_l (x) a_{l-1}   (reduction over positions)        warp-level TF32 MMAs m16n8k8: M = out channel, N = (tap, in
//                                                                 channel), K = position; accumulators stay in REGISTERS for
//                                                                 the whole kernel (a warp owns the same tiles in every group)
//   g_{l-1} = W_l^T * dY_l      (full correlation)                M = in channel, N = input position, K = (tap, out channel);
//                                                                 A = fragment-packed weight images resident in shared memory
//
// Why mma.sync and not tcgen05 here: the tiles are 32 x (32 ks) with a reduction of 8 VT positions per pass -- below the
// M = 64 minimum of tcgen05.mma, and each would pay a TMEM round trip; at these shapes the warp-level MMA with operands read
// straight from the activation planes (bank-conflict-free strides) is the tensor-core instruction that fits.
// Gradients use single-pass TF32 operands rounded to nearest with fp32 accumulation, the same contract as the read path's
// tensor-core backward (pmt_tc_bwd.cu; tests/test_backward_tc_gpu.py).  Every sum has a fixed order: bitwise reproducible.
#include <cstring>

#include "pmt_call.h"

namespace pmt {
namespace cnnbwd {

__host__ __device__ __forceinline__ int w_index(const BLayer& Ly, int co, int ci, int t) {
  if (Ly.is_linear) return Ly.w_off + co * Ly.op_in_ch + (Ly.flat_len > 1 ? ci * Ly.flat_len + t : ci);
  return Ly.w_off + (co * Ly.op_in_ch + ci) * Ly.ks + t;
}

// Data-gradient images: for (tap t, k-step kc over out channels, m-tile m over in channels) the A fragment of
// A[ci][co] = W[co][ci][t], 128 floats: lane * 4 + {(co, ci), (co, ci + 8), (co + 4, ci), (co + 4, ci + 8)} with
// co = 8 kc + lane % 4, ci = 16 m + lane / 4.
__global__ void pack_cnn_bwd_kernel(const __grid_constant__ BPlan BP, const float* __restrict__ w, float* __restrict__ image) {
  const BLayer& Ly = BP.layer[blockIdx.x];
  if (blockIdx.x == 0) return;
  const int n = Ly.ks * Ly.Cout8 * Ly.Mt_d * 128;
  for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < n; idx += gridDim.y * blockDim.x) {
    const int r = idx & 3, lane = (idx >> 2) & 31, frag = idx >> 7;
    const int m = frag % Ly.Mt_d, kc = (frag / Ly.Mt_d) % Ly.Cout8, t = frag / (Ly.Mt_d * Ly.Cout8);
    const int co = kc * 8 + (lane & 3) + ((r & 2) ? 4 : 0), ci = m * 16 + (lane >> 2) + ((r & 1) ? 8 : 0);
    const float v = (co < Ly.Cout && ci < Ly.Cin) ? w[w_index(Ly, co, ci, t)] : 0.f;
    image[Ly.img_off + idx] = rna_tf32(v);
  }
}

// What a weight-gradient unit needs from its layer, in registers
struct WgLayer {
  int first, ks, Cin8, kpv, lm, lpg, ldy, L_in, ld_a, a_smem;
};
// Constant rows behind the planes / codes: the bias tile's B operand (ones for column 0 of the tile, i.e. for the lanes
// with lane / 4 == 0) and the operand of the unused tiles of a unit's last group (zeros), both read with stride 0.
constexpr int CONST_ROW = 16;               // floats (bytes for the codes) per constant row
constexpr int CODE_ONE = 77, CODE_NONE = 78;

template <bool FIRST>
__device__ __forceinline__ void wgrad_unit(const WgLayer& Ly, int VT, int codes_stride, int const_off, const Unit& U, float (&acc)[NT][4],
                                           const float* __restrict__ dY, const float* __restrict__ planes,
                                           const unsigned char* __restrict__ codes, int nv, int lane) {
  const int gid = lane >> 2, tig = lane & 3;
  const int bias_tile = Ly.ks * Ly.Cin8;
  int rowj[NT], mulj[NT], cj[NT];   // B row offset, 1 (walks with the position) or 0 (constant row), one-hot channel (FIRST)
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int nt = U.nt0 + j;
    if (j >= U.cnt) { rowj[j] = const_off + CONST_ROW; mulj[j] = 0; cj[j] = CODE_ONE; }                              // zeros
    else if (nt == bias_tile) { rowj[j] = const_off + (gid == 0 ? 0 : CONST_ROW); mulj[j] = 0; cj[j] = CODE_ONE; }   // ones in column 0
    else {
      const int t = nt / Ly.Cin8, ct = nt - t * Ly.Cin8, n = ct * 8 + gid;
      mulj[j] = 1; cj[j] = n >> 1;
      // first layer: the codes of haplotype h = n & 1, compared with channel c = n >> 1 below
      rowj[j] = FIRST ? (n & 1) * VT * codes_stride + tig + t : Ly.a_smem + n * Ly.ld_a + tig + t;
    }
    if (mulj[j] == 0) rowj[j] += tig;
  }
  const float* a_r0 = dY + (U.m * 16 + gid) * Ly.ldy + Ly.lm + tig;
  const float* a_r1 = a_r0 + 8 * Ly.ldy;
  const int cstep = FIRST ? codes_stride : Ly.L_in;
  for (int v = 0; v < nv; ++v) {
    for (int kk = 0; kk < Ly.kpv; ++kk) {
      const int base = v * Ly.lpg + kk * 8, boff = v * cstep + kk * 8;
      float a[4];
      a[0] = a_r0[base]; a[1] = a_r1[base]; a[2] = a_r0[base + 4]; a[3] = a_r1[base + 4];
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        float b0, b1;
        if (FIRST) {
          const unsigned char* cp = codes + rowj[j] + boff * mulj[j];
          b0 = cp[0] == cj[j] ? 1.f : 0.f; b1 = cp[4] == cj[j] ? 1.f : 0.f;
        } else {
          const float* bp = planes + rowj[j] + boff * mulj[j];
          b0 = bp[0]; b1 = bp[4];
        }
        mma_tf32(acc[j], a, b0, b1);
      }
    }
  }
}

// dY_l = route(g_l through the fused pool) * act'(a_l), with its zero margins.  MODE 0: no pool, 1: MaxPool(2, 1), 2: MaxPool(2, 2);
// GLOBAL: the output layer (g and the activation come from global memory).
template <int MODE, bool GLOBAL>
__device__ __forceinline__ void make_dY(float* __restrict__ dY, const float* __restrict__ gin, int ld_gin, const float* __restrict__ ap, int ld_an,
                                        const unsigned char* __restrict__ bp, int VT, int nv, int Cout, int lpg, int ldy, int lm, int L_out,
                                        int Lp, int selu, const float* __restrict__ d_out, const float* __restrict__ y_out, int out_w) {
  const int tid = threadIdx.x;
  const int bcols = VT * Lp, row_el = VT * lpg, n_el = Cout * row_el;
  // (co, v, x) of element tid, then steps of THREADS elements without divisions
  int co = tid / row_el, rem = tid - co * row_el;
  int v = rem / lpg, x = rem - v * lpg;
  const int dco = THREADS / row_el, drem = THREADS - dco * row_el, dv = drem / lpg, dx = drem - dv * lpg;
  const float sa = selu ? SELU_SCALE : 0.f, sb = selu ? SELU_SCALE * SELU_ALPHA : 1.f, sc = selu ? SELU_SCALE : 1.f;   // act' = a > 0 ? sc : sa a + sb
  for (int i = tid; i < n_el; i += THREADS) {
    const int q = x - lm;
    float val = 0.f;
    if (q >= 0 && q < L_out && v < nv) {
      // pooled positions that route into conv position q.  MaxPool(2, 1): q (first element of its window) and q - 1 (second);
      // MaxPool(2, 2): q >> 1 when q's parity is the winner's
      const int p0 = MODE == 2 ? q >> 1 : q;
      const int boff = (co >> 3) * bcols + v * Lp, bsh = co & 7;
      if (p0 < Lp) {
        const int want = MODE == 2 ? q & 1 : 0;
        const int b = MODE ? (bp[boff + p0] >> bsh) & 1 : 0;
        if (b == want) {
          float g, a;
          if (GLOBAL) {
            const long long o = (long long)v * out_w + co;
            g = __ldg(d_out + o); a = selu ? __ldg(y_out + o) * (1.f / SELU_SCALE) : 1.f;
          } else {
            g = gin[co * ld_gin + v * Lp + p0]; a = ap[co * ld_an + v * Lp + p0];
          }
          val = g * (a > 0.f ? sc : fmaf(sa, a, sb));
        }
      }
      if (MODE == 1 && q >= 1 && ((bp[boff + q - 1] >> bsh) & 1)) {
        const float g = gin[co * ld_gin + v * Lp + q - 1], a = ap[co * ld_an + v * Lp + q - 1];
        val += g * (a > 0.f ? sc : fmaf(sa, a, sb));
      }
    }
    dY[co * ldy + v * lpg + x] = rna_tf32(val);
    co += dco; v += dv; x += dx;
    if (x >= lpg) { x -= lpg; v += 1; }
    if (v >= VT) { v -= VT; co += 1; }
  }
}

__global__ void __launch_bounds__(THREADS, 1)
cnn_backward_mma_kernel(const __grid_constant__ BPlan BP_param, const float* __restrict__ image_g, const void* __restrict__ haps, int hap_kind,
                        long long hap_stride, int n_variants, const float* __restrict__ save, const float* __restrict__ info_seq,
                        const float* __restrict__ d_info_seq, int out_w, int d_info, float* __restrict__ partials, int n_params) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  BPlan* BPs = reinterpret_cast<BPlan*>(smem_raw);
  float* img = reinterpret_cast<float*>(smem_raw + ((sizeof(BPlan) + 15) & ~size_t(15)));
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  {
    const int* src = reinterpret_cast<const int*>(&BP_param);
    for (int i = tid; i < (int)(sizeof(BPlan) / sizeof(int)); i += THREADS) reinterpret_cast<int*>(BPs)[i] = src[i];
  }
  __syncthreads();
  const BPlan& BP = *BPs;
  // [images][planes x 2][dY][g][window bits x 2][codes x 2]: the activations of the NEXT group are fetched (cp.async) while
  // this group is processed
  float* planes_all = img + BP.img_total;
  float* crow = planes_all + 2 * BP.a_total;            // [ones | zeros] rows of CONST_ROW floats (wgrad_unit)
  float* dY = crow + 2 * CONST_ROW;
  float* gbuf = dY + BP.dy_floats;
  unsigned char* bits_all = reinterpret_cast<unsigned char*>(gbuf + BP.g_floats);
  unsigned char* codes_all = bits_all + 2 * BP.bits_bytes;
  const int VT = BP.VT, nL = BP.n_layers, G = BP.G, L0 = BP.L0, codes_stride = BP.codes_stride;
  const int codes_bytes = 2 * VT * codes_stride;
  for (int i = tid; i < BP.img_total / 4; i += THREADS) reinterpret_cast<float4*>(img)[i] = __ldg(reinterpret_cast<const float4*>(image_g) + i);
  // everything a fragment load may touch beyond the valid data must be finite (it meets zeros)
  for (int i = tid; i < 2 * BP.a_total + 2 * CONST_ROW + BP.dy_floats + BP.g_floats; i += THREADS) planes_all[i] = 0.f;
  for (int i = tid; i < 2 * codes_bytes; i += THREADS) codes_all[i] = 255;
  __syncthreads();
  if (tid < 2 * CONST_ROW) {
    crow[tid] = tid < CONST_ROW ? 1.f : 0.f;
    codes_all[2 * codes_bytes + tid] = tid < CONST_ROW ? CODE_ONE : CODE_NONE;
  }

  float acc[SLOTS][NT][4];
#pragma unroll
  for (int s = 0; s < SLOTS; ++s)
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[s][j][r] = 0.f;

  const int gid = lane >> 2, tig = lane & 3;
  const int n_groups = (n_variants + VT - 1) / VT;

  // ---- a group's saved activations a_{l-1} (raw: the SELU scale of the producing layer is applied where they are used),
  //      window bits and haplotype codes into buffer `buf` ----
  auto fetch = [&](int grp, int buf) {
    const int v0 = grp * VT, nv = min(VT, n_variants - v0);
    const int gf = v0 / G, sub = v0 - gf * G;
    const float* sg = save + (size_t)gf * BP.group_floats;
    float* planes = planes_all + buf * BP.a_total;
    for (int l = 1; l < nL; ++l) {
      const BLayer& Ly = BP.layer[l];
      const int cols4 = (VT * Ly.L_in) >> 2, gcols = G * Ly.L_in, ok_bytes = nv * Ly.L_in * 4, ld_a = Ly.ld_a, n4 = Ly.Cin * cols4;
      const float* src = sg + Ly.save_in + sub * Ly.L_in;
      float* dst = planes + Ly.a_smem;
      int c = tid / cols4, k = tid - c * cols4;
      const int dc = THREADS / cols4, dk = THREADS - dc * cols4;
      for (int i = tid; i < n4; i += THREADS) {
        const int left = ok_bytes - k * 16;
        cp_async16_zfill(dst + c * ld_a + k * 4, src + c * gcols + k * 4, left >= 16 ? 16 : (left > 0 ? left : 0));
        c += dc; k += dk;
        if (k >= cols4) { k -= cols4; c += 1; }
      }
    }
    unsigned char* bits = bits_all + buf * BP.bits_bytes;
    for (int l = 0; l < nL; ++l) {
      const BLayer& Ly = BP.layer[l];
      if (Ly.save_bits < 0) continue;
      const int cols = VT * Ly.L_pool, gcols = G * Ly.L_pool, ok = nv * Ly.L_pool;
      const unsigned char* src = reinterpret_cast<const unsigned char*>(sg + Ly.save_bits) + sub * Ly.L_pool;
      for (int i = tid; i < 4 * cols; i += THREADS) {
        const int cq = i / cols, col = i - cq * cols;
        bits[Ly.bits_smem + i] = col < ok ? __ldg(src + cq * gcols + col) : (unsigned char)0;
      }
    }
    unsigned char* codes = codes_all + buf * codes_bytes;
    for (int i = tid; i < VT * 2 * L0; i += THREADS) {
      const int v = i / (2 * L0), hp = i - v * 2 * L0, h = hp / L0, p = hp - h * L0;
      int code = 255;
      if (v < nv) {
        const long long off = (long long)(v0 + v) * hap_stride + hp;
        code = hap_kind == PMT_I64 ? (int)reinterpret_cast<const long long*>(haps)[off] : (int)reinterpret_cast<const short*>(haps)[off];
      }
      codes[(h * VT + v) * codes_stride + p] = (unsigned char)(code & 255);
    }
    cp_async_commit();
  };

  if ((int)blockIdx.x < n_groups) fetch(blockIdx.x, 0);
  int buf = 0;
  for (int grp = blockIdx.x; grp < n_groups; grp += gridDim.x, buf ^= 1) {
    const int v0 = grp * VT, nv = min(VT, n_variants - v0);
    const float* planes = planes_all + buf * BP.a_total;
    const unsigned char* bits = bits_all + buf * BP.bits_bytes;
    const unsigned char* codes = codes_all + buf * codes_bytes;
    cp_async_wait_all();
    __syncthreads();   // this group's buffers are complete; every warp is done with the previous group's
    if (grp + (int)gridDim.x < n_groups) fetch(grp + gridDim.x, buf ^ 1);

    for (int l = nL - 1; l >= 0; --l) {
      const BLayer& LyS = BP.layer[l];
      const int lpg = LyS.lpg, ldy = LyS.ldy, lm = LyS.lm, L_out = LyS.L_out, Lp = LyS.L_pool, Cout = LyS.Cout;
      // ---- dY_l: the gradient through the fused pool and the activation, written with its zero margins ----
      {
        const BLayer& Nx = BP.layer[l + 1 < nL ? l + 1 : l];
        const float* ap = planes + Nx.a_smem;
        const unsigned char* bp = bits + LyS.bits_smem;
        const float* d_out = d_info_seq + (long long)v0 * out_w + d_info;
        const float* y_out = info_seq + (long long)v0 * out_w + d_info;
        if (LyS.to_global) make_dY<0, true>(dY, gbuf, 0, ap, 0, bp, VT, nv, Cout, lpg, ldy, lm, L_out, Lp, LyS.selu, d_out, y_out, out_w);
        else if (LyS.dup) make_dY<1, false>(dY, gbuf, Nx.ld_g, ap, Nx.ld_a, bp, VT, nv, Cout, lpg, ldy, lm, L_out, Lp, LyS.selu, d_out, y_out, out_w);
        else if (LyS.pool2) make_dY<2, false>(dY, gbuf, Nx.ld_g, ap, Nx.ld_a, bp, VT, nv, Cout, lpg, ldy, lm, L_out, Lp, LyS.selu, d_out, y_out, out_w);
        else make_dY<0, false>(dY, gbuf, Nx.ld_g, ap, Nx.ld_a, bp, VT, nv, Cout, lpg, ldy, lm, L_out, Lp, LyS.selu, d_out, y_out, out_w);
      }
      __syncthreads();
      // ---- weight gradient: the units this warp owns ----
      {
        WgLayer W;
        W.first = LyS.first; W.ks = LyS.ks; W.Cin8 = LyS.Cin8; W.kpv = LyS.kpv; W.lm = lm; W.lpg = lpg; W.ldy = ldy;
        W.L_in = LyS.L_in; W.ld_a = LyS.ld_a; W.a_smem = LyS.a_smem;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
          const int u = warp + WARPS * s;
          if (u < BP.n_units && BP.unit[u].layer == l) {
            const Unit U = BP.unit[u];
            if (W.first) wgrad_unit<true>(W, VT, codes_stride, 2 * codes_bytes - buf * codes_bytes, U, acc[s], dY, planes_all, codes_all + buf * codes_bytes, nv, lane);
            else wgrad_unit<false>(W, VT, codes_stride, 2 * BP.a_total - buf * BP.a_total, U, acc[s], dY, planes, codes, nv, lane);
          }
        }
      }
      // ---- data gradient g_{l-1}[ci][v, q'] = sum_{t, co} W[co][ci][t] dY_l[co][v, q' - t] ----
      if (l > 0) {
        const int Mt_d = LyS.Mt_d, ks = LyS.ks, Cout8 = LyS.Cout8, npv = LyS.npv, L_in = LyS.L_in, ld_g = LyS.ld_g, Cin = LyS.Cin;
        const int fstep = Mt_d * 128;
        for (int u = warp; u < Mt_d * VT; u += WARPS) {
          const int m = u / VT, v = u - m * VT;
          if (v >= nv) continue;
          float d[MAX_NPV][4];
#pragma unroll
          for (int j = 0; j < MAX_NPV; ++j) { d[j][0] = 0.f; d[j][1] = 0.f; d[j][2] = 0.f; d[j][3] = 0.f; }
          const float* fr = img + LyS.img_off + m * 128 + lane * 4;
          const float* yv = dY + tig * ldy + v * lpg + lm + gid;
          for (int t = 0; t < ks; ++t) {
            const float* yk = yv - t;
            for (int kc = 0; kc < Cout8; ++kc) {
              const float4 af = *reinterpret_cast<const float4*>(fr);
              fr += fstep;
              const float a[4] = {af.x, af.y, af.z, af.w};
#pragma unroll
              for (int j = 0; j < MAX_NPV; ++j)
                if (j < npv) mma_tf32(d[j], a, yk[j * 8], yk[j * 8 + 4 * ldy]);
              yk += 8 * ldy;
            }
          }
          const int ci0 = m * 16 + gid, ci1 = ci0 + 8;
#pragma unroll
          for (int j = 0; j < MAX_NPV; ++j) {
            if (j >= npv) continue;
            const int q0 = j * 8 + 2 * tig;
            float* o0 = gbuf + ci0 * ld_g + v * L_in + q0;
            float* o1 = gbuf + ci1 * ld_g + v * L_in + q0;
            if (ci0 < Cin) { if (q0 < L_in) o0[0] = d[j][0]; if (q0 + 1 < L_in) o0[1] = d[j][1]; }
            if (ci1 < Cin) { if (q0 < L_in) o1[0] = d[j][2]; if (q0 + 1 < L_in) o1[1] = d[j][3]; }
          }
        }
      }
      __syncthreads();
    }
  }

  // ---- flush: every parameter entry has exactly one owner (unit, lane, register) ----
  float* part = partials + (size_t)blockIdx.x * n_params;
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int u = warp + WARPS * s;
    if (u >= BP.n_units) continue;
    const Unit U = BP.unit[u];
    const BLayer& Ly = BP.layer[U.layer];
    const int bias_tile = Ly.ks * Ly.Cin8;
    const int co0 = U.m * 16 + gid, co1 = co0 + 8;
    const float s_in = Ly.s_in;   // the planes hold the saved activations without the producing layer's SELU scale
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      if (j >= U.cnt) continue;
      const int nt = U.nt0 + j;
      if (nt == bias_tile) {
        if (tig == 0 && Ly.b_off >= 0) {
          if (co0 < Ly.Cout) red_add(part + Ly.b_off + co0, acc[s][j][0]);
          if (co1 < Ly.Cout) red_add(part + Ly.b_off + co1, acc[s][j][2]);
        }
        continue;
      }
      const int t = nt / Ly.Cin8, ct = nt - t * Ly.Cin8;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int co = (r & 2) ? co1 : co0, ci = ct * 8 + 2 * tig + (r & 1);
        if (co < Ly.Cout && ci < Ly.Cin) red_add(part + w_index(Ly, co, ci, t), s_in * acc[s][j][r]);
      }
    }
  }
}

}  // namespace cnnbwd
}  // namespace pmt

// ================================================================================================
// host side
// ================================================================================================
using namespace pmt;
using namespace pmt::cnnbwd;

static int pad_mod(int n, int r, int m) {   // smallest ld >= n with ld == r (mod m)
  int ld = n;
  while (ld % m != r) ++ld;
  return ld;
}

// Layer program of the backward from the forward's; false: outside this kernel's envelope (the FP32 SIMT kernel runs).
bool pmt_build_cnn_bwd_plan(const pmt::Plan& P, const cnntc::Plan& T, BPlan* out) {
  BPlan& B = *out;
  memset(&B, 0, sizeof(B));
  cnntc::SaveLayout SL;
  pmt_cnn_save_layout(T, &SL);
  const PmtModelDesc& d = P.d;
  B.n_layers = T.n_layers; B.G = T.G; B.group_floats = SL.group_floats; B.L0 = T.L0;
  if (T.n_layers < 2 || T.n_layers > MAXL) return false;
  for (int vt : {8, 4}) {
    if (T.G % vt != 0) continue;
    B.VT = vt; B.inv_vt = 65536 / vt + (65536 % vt ? 1 : 0);
    int img = 0, a_tot = 0, dy = 0, gf = 0, bits = 0;
    bool ok = true;
    for (int l = 0; l < T.n_layers && ok; ++l) {
      const cnntc::Layer& F = T.layer[l];
      const PmtCnnOp& op = d.cnn_ops[F.op];
      BLayer& Ly = B.layer[l];
      memset(&Ly, 0, sizeof(Ly));
      Ly.first = F.first; Ly.is_linear = F.is_linear; Ly.flat_len = F.flat_len; Ly.to_global = F.to_global;
      Ly.Cin = F.first ? cnntc::C0 : F.in_ch; Ly.Cout = F.out_ch; Ly.ks = F.ksize;
      Ly.L_in = F.L_in; Ly.L_out = F.L_out; Ly.L_pool = F.L_pool;
      Ly.dup = F.dup; Ly.pool2 = F.pool2; Ly.selu = F.act == PMT_ACT_SELU;
      Ly.w_off = op.w_off; Ly.b_off = op.b_off; Ly.op_in_ch = op.in_ch;
      Ly.s_in = F.scale_in ? SELU_SCALE : 1.f;
      if (F.first && (Ly.Cin != cnntc::C0 || op.in_ch != cnntc::C0)) ok = false;
      if (Ly.Cin > 32 || Ly.Cout > 32 || Ly.ks < 1) ok = false;
      if (Ly.L_out != Ly.L_in - Ly.ks + 1) ok = false;
      if (F.to_global != (l == T.n_layers - 1)) ok = false;
      Ly.Cin8 = (Ly.Cin + 7) / 8; Ly.Cout8 = (Ly.Cout + 7) / 8;
      Ly.Mt_w = (Ly.Cout + 15) / 16; Ly.Mt_d = (Ly.Cin + 15) / 16;
      Ly.kpv = (Ly.L_out + 7) / 8; Ly.npv = (Ly.L_in + 7) / 8;
      if (l > 0 && Ly.npv > MAX_NPV) ok = false;
      Ly.lm = Ly.ks - 1;
      int right = Ly.kpv * 8 - Ly.L_out;
      if (right < Ly.ks - 1) right = Ly.ks - 1;
      Ly.lpg = Ly.lm + Ly.L_out + right;
      if (Ly.lpg > 32) ok = false;                         // one lane per position of a (channel, variant) row
      Ly.ldy = pad_mod(vt * Ly.lpg + 40, 8, 16);           // slack: the data gradient's padded columns read past the last variant
      if (32 * Ly.ldy > dy) dy = 32 * Ly.ldy;
      Ly.save_bits = SL.bits_off[l];
      if ((F.dup || F.pool2) && Ly.save_bits < 0) ok = false;
      if (Ly.save_bits >= 0) { Ly.bits_smem = bits; bits += 4 * vt * Ly.L_pool; }
      if (l > 0) {
        Ly.save_in = SL.a_off[l - 1];
        if (Ly.save_in < 0) ok = false;
        if (B.layer[l - 1].Cout != Ly.Cin || B.layer[l - 1].L_pool != Ly.L_in) ok = false;
        Ly.ld_a = pad_mod(vt * Ly.L_in + 8, 4, 8);          // == 4 (mod 8): the B fragment's 8 rows x 4 columns hit 32 banks
        Ly.a_smem = a_tot; a_tot += Ly.Cin8 * 8 * Ly.ld_a;
        Ly.ld_g = pad_mod(vt * Ly.L_in, 8, 16);
        if (Ly.Cin8 * 8 * Ly.ld_g > gf) gf = Ly.Cin8 * 8 * Ly.ld_g;
        Ly.img_off = img; img += Ly.ks * Ly.Cout8 * Ly.Mt_d * 128;
      }
    }
    if (!ok) return false;
    // weight-gradient units in processing order (last layer first), so that a layer's units sit on different warps
    B.n_units = 0;
    for (int l = T.n_layers - 1; l >= 0 && ok; --l) {
      const BLayer& Ly = B.layer[l];
      const int n_tiles = Ly.ks * Ly.Cin8 + 1;   // + the bias tile
      for (int m = 0; m < Ly.Mt_w && ok; ++m)
        for (int nt0 = 0; nt0 < n_tiles; nt0 += NT) {
          if (B.n_units >= MAX_UNITS) { ok = false; break; }
          Unit& U = B.unit[B.n_units++];
          U.layer = l; U.m = m; U.nt0 = nt0; U.cnt = n_tiles - nt0 < NT ? n_tiles - nt0 : NT;
        }
    }
    if (!ok) return false;
    B.img_total = (img + 3) & ~3; B.a_total = (a_tot + 3) & ~3; B.dy_floats = (dy + 3) & ~3; B.g_floats = (gf + 3) & ~3;
    B.bits_bytes = (bits + 15) & ~15;
    B.codes_stride = ((B.layer[0].kpv * 8 + B.layer[0].ks + 8 + T.L0) + 3) & ~3;
    const size_t smem = ((sizeof(BPlan) + 15) & ~size_t(15)) + (size_t)(B.img_total + 2 * B.a_total + B.dy_floats + B.g_floats) * sizeof(float) +
                        2 * B.bits_bytes + 2 * 2 * vt * B.codes_stride + 2 * CONST_ROW * (sizeof(float) + 1) + 64;
    B.smem_bytes = (int)smem;
    if (smem <= 227 * 1024) return true;
  }
  return false;
}

// the training forward runs the SAVE variant over the whole batch (pmt_forward_train); `save`: the CNN part of the saved
// buffer
int pmt_cnn_forward_train(const CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq, unsigned char* image,
                          float* save, cudaStream_t st) {
  if (pmt_pack_cnn_tc_images(C.P, C.C, weights, image, st)) return 1;
  return pmt_launch_cnn_tc_save(C.P, C.C, weights, batch, 0, batch->n_variants, info_seq, image, save, C.n_sm, st);
}

int pmt_launch_cnn_backward_mma(const CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq, const float* d_info_seq,
                                float* partials, const CnnBwdBuffers& W, cudaStream_t st, const float* saved) {
  const pmt::Plan& P = C.P;
  const cnntc::Plan& T = C.C;
  const BPlan& B = C.CB;
  float* save = W.save;
  // weight images: the forward's (split precision; only for the recompute) and the data gradient's
  if (!saved && pmt_pack_cnn_tc_images(P, T, weights, W.fwd_image, st)) return 1;
  pack_cnn_bwd_kernel<<<dim3(B.n_layers, 8), 256, 0, st>>>(B, weights, W.bwd_image);
  PMT_CUDA(cudaFuncSetAttribute(cnn_backward_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, B.smem_bytes));
  const int out_w = P.d.d_info + P.d.d_seq;
  const size_t esz = batch->hap_kind == PMT_I64 ? 8 : 2;
  const int chunk = saved ? batch->n_variants : PMT_CNN_BWD_CHUNK;   // saved by the training forward: the whole batch at once
  for (int v_first = 0; v_first < batch->n_variants; v_first += chunk) {
    const int n = batch->n_variants - v_first < chunk ? batch->n_variants - v_first : chunk;
    if (saved) save = const_cast<float*>(saved);
    else if (pmt_launch_cnn_tc_save(P, T, weights, batch, v_first, n, info_seq, W.fwd_image, save, C.n_sm, st)) return 1;
    const int n_groups = (n + B.VT - 1) / B.VT;
    int grid = n_groups < C.n_sm ? n_groups : C.n_sm;
    if (grid > PMT_PARTIAL_CTAS) grid = PMT_PARTIAL_CTAS;
    const void* haps = reinterpret_cast<const unsigned char*>(batch->haplotypes) + (size_t)v_first * batch->hap_stride * esz;
    cnn_backward_mma_kernel<<<grid, THREADS, B.smem_bytes, st>>>(B, W.bwd_image, haps, batch->hap_kind, batch->hap_stride, n, save,
                                                                 info_seq + (size_t)v_first * out_w, d_info_seq + (size_t)v_first * out_w, out_w,
                                                                 P.d.d_info, partials, P.d.n_params);
  }
  return 0;
}
