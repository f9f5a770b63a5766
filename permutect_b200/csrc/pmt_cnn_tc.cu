// Tensor-core (tcgen05 / TMEM) forward of the haplotype CNN (batch.py:115-130 one-hot + dna_sequence_convolution.py:57-111).
//
// A 1-D convolution over G variants is one GEMM whose rows are the FLAT positions j = v * L_in + p of the group:
//     out[j][co] = sum_t sum_ci in[j + t][ci] * W[co][ci][t]
// i.e. ksize accumulating MMAs whose A operand is the SAME activation buffer shifted by t rows.  Activations live in
// shared memory position-major in the no-swizzle K-major canonical layout "[16-byte channel chunk][row][4 floats]"
// (8 planes of PLANE_ROWS rows): core matrices of 8 rows x 16 B are contiguous, 8-row groups are 128 B apart
// (SBO) and K-adjacent core matrices one plane apart (LBO), so a shift by t rows is the start address + 16 t bytes.
// Rows j whose window straddles two variants compute garbage that nobody reads.
//
//   warps 0-7  epilogue: thread = output row (TMEM lane) of a 128-row chunk; even chunks -> warps 0-3, odd -> warps 4-7.
//              bias, max-pool, SELU, hi/lo split, compaction to the next layer's row stride, IN PLACE (a compacted row
//              index never exceeds the source row index, and chunks complete in order).
//   warp  8    MMA issuer: per layer, all chunks back to back into separate TMEM accumulators, one commit per chunk.
//
// The first conv reads the one-hot input as an im2col row [onehot(p) | onehot(p+1) | ...] (exact in TF32, no lo pass);
// a MaxPool(kernel 2, stride 1) that follows it is fused by computing the conv at p and p+1 side by side in N.
// MaxPool(2, 2) elsewhere is a lane shuffle (row strides are even).  Flatten + Linear is a conv whose kernel covers
// the whole remaining length.  SELU scales are folded into the consuming weights.  Precision modes as pmt_tc.cu.
// Inference splits the layers: this kernel runs the head and hands its last activation to hap_cnn_tail_kernel through
// global memory, so the short tail layers (few rows per group, a full MMA -> epilogue round trip each) run as dense layers
// over 128 variants.  The training forward (SAVE) runs every layer here.
#include <cstring>

#include "pmt_call.h"

namespace pmt {
namespace cnntc {

using namespace pmt::tc;

// Split-precision scheme (PASSES == 3): the weight image stacks [W_hi ; W_lo] along N, so ONE MMA of width 2N computes
// A_hi.W_hi (columns [0, N)) and A_hi.W_lo (columns [N, 2N)) from a single read of the A rows -- operand fetch from shared
// memory, not the tensor pipe, bounds these small-N MMAs -- and a second MMA of width N adds A_lo.W_hi to columns [0, N).
// The epilogue sums the two column ranges.  PASSES == 1 uses the W_hi rows only.
//
// shifted-window conv: taps x 4 k-steps.  The tap loop is a warp-uniform runtime loop (no jump table: an indirect
// branch would push every descriptor out of the uniform registers); inside a tap all offsets are compile-time constants.
template <int PASSES>
__device__ __forceinline__ void issue_shifted(int taps, unsigned d, unsigned a_hi, unsigned a_lo, unsigned b) {
  constexpr int R = 64;   // image rows per plane: 32 hi + 32 lo
#pragma unroll 1
  for (int t = 0; t < taps; ++t) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const unsigned ao = (unsigned)(2 * ks * (PLANE_BYTES / 16));
      const unsigned bo = (unsigned)(2 * ks * R);
      const unsigned acc = (ks == 0) ? (t > 0 ? 1u : 0u) : 1u;
      if (PASSES == 3) {
        mma_ss_desc_lo<make_idesc(64)>(d, a_hi + ao, b + bo, acc);
        mma_ss_desc_lo<make_idesc(32)>(d, a_lo + ao, b + bo, 1u);
      } else {
        mma_ss_desc_lo<make_idesc(32)>(d, a_hi + ao, b + bo, acc);
      }
    }
    a_hi += 1; a_lo += 1; b += 8 * R;
  }
}
// first conv: one-hot im2col rows (exact: no A lo pass), K = 8 * KS columns over consecutive planes
template <int N, int PASSES>
__device__ __forceinline__ void issue_first(int ksteps, unsigned d, unsigned a, unsigned b) {
  constexpr int R = 2 * N;
  constexpr unsigned idesc = make_idesc(PASSES == 3 ? 2 * N : N);
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    if (ks < ksteps) {
      const unsigned ao = (unsigned)(2 * ks * (PLANE_BYTES / 16)), bo = (unsigned)(2 * ks * R);
      mma_ss_desc_lo<idesc>(d, a + ao, b + bo, ks != 0 ? 1u : 0u);
    }
  }
}

struct ItemDev {   // per-item MMA operands, computed once per CTA
  unsigned a_hi, a_lo, b, d;
  int first, count, N, need;
};

struct EpiItem {   // per-item epilogue constants (three 16-byte shared loads)
  int flags, lo_col, tmem_col, bias_off;
  int inv_L, L_in, L_pool, L_next;
  int row0, out_ch, save_a, save_bits;   // SAVE: float offsets inside a group's block of the save buffer (-1: none)
};
constexpr int F_DUP = 1, F_POOL2 = 2, F_GLOBAL = 4, F_SELU = 8, F_TAIL = 16;

struct Bars {
  EpiItem epi[MAX_ITEMS];
  unsigned long long done_bar[MAX_ITEMS + 1];   // [0]: im2col rows written; [1 + i]: epilogue of item i finished (16 warps)
  unsigned long long acc_bar[MAX_ITEMS];        // accumulator of item i complete (tcgen05.commit)
  ItemDev item[MAX_ITEMS];
  unsigned tmem_base;
  int pad_;
};
constexpr int CNN_TMEM_COLS = MAX_CHUNKS * CHUNK_COLS;   // one accumulator per chunk

template <int PASSES, bool SAVE>
__global__ void __launch_bounds__(THREADS, 1)
hap_cnn_tc_kernel(const __grid_constant__ Plan TP, const unsigned char* __restrict__ image, const float* __restrict__ wflat,
                  const __grid_constant__ PmtModelDesc D, const void* __restrict__ haps, int hap_kind, long long hap_stride,
                  int n_variants, float* __restrict__ info_seq,
                  const __grid_constant__ SaveLayout SL, float* __restrict__ save, float* __restrict__ tail_buf) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* p = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const unsigned act = smem_addr(p); p += 2 * BUF_BYTES;                 // hi buffer, then lo buffer (planes 8..15)
  unsigned char* img_s = p; p += TP.image_bytes;
  float* bias_s = reinterpret_cast<float*>(p); p += MAX_LAYERS * 32 * sizeof(float);
  Bars* S = reinterpret_cast<Bars*>((reinterpret_cast<uintptr_t>(p) + 15) & ~uintptr_t(15));

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int lane = tid & 31;
  const int n_layers = TP.n_layers, n_items = TP.n_items, G = TP.G, L0 = TP.L0;

  if (tid == 0) {
    for (int i = 0; i <= n_items; ++i) mbar_init(smem_addr(&S->done_bar[i]), EPI_WARPS);
    for (int i = 0; i < n_items; ++i) mbar_init(smem_addr(&S->acc_bar[i]), 1);
    fence_mbar_init();
  }
  // resident weight images (no-swizzle K-major planes, built by pack_cnn_tc_kernel) and biases
  for (int i = tid; i < TP.image_bytes / 16; i += THREADS)
    reinterpret_cast<uint4*>(img_s)[i] = __ldg(reinterpret_cast<const uint4*>(image) + i);
  for (int i = tid; i < n_layers * 32; i += THREADS) {
    const Layer& Ly = TP.layer[i / 32];
    const int n = i % 32, b_off = D.cnn_ops[Ly.op].b_off;
    bias_s[i] = (n < Ly.out_ch && b_off >= 0) ? __ldg(wflat + b_off + n) : 0.f;
  }
  if (warp == MMA_WARP) tmem_alloc<CNN_TMEM_COLS>(smem_addr(&S->tmem_base));
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = __shfl_sync(0xffffffffu, S->tmem_base, 0);
  const int n_groups = (n_variants + G - 1) / G;
  if (tid < n_items) {
    const Item& I = TP.item[tid];
    const Layer& Ly = TP.layer[I.layer];
    ItemDev& o = S->item[tid];
    o.a_hi = desc_lo(act + I.chunk * 128 * 16, PLANE_BYTES);
    o.a_lo = desc_lo(act + BUF_BYTES + I.chunk * 128 * 16, PLANE_BYTES);
    o.b = desc_lo(smem_addr(img_s) + Ly.img_off, 2 * Ly.N * 16);
    o.d = tmem_base + I.chunk * CHUNK_COLS;
    o.first = Ly.first; o.count = Ly.first ? Ly.ksteps : Ly.taps; o.N = Ly.N; o.need = I.need;
    EpiItem& e = S->epi[tid];
    e.flags = (Ly.dup ? F_DUP : 0) | (Ly.pool2 ? F_POOL2 : 0) | (Ly.to_global ? F_GLOBAL : 0) | (Ly.act == PMT_ACT_SELU ? F_SELU : 0) |
              (Ly.to_tail ? F_TAIL : 0);
    e.lo_col = Ly.N; e.tmem_col = I.chunk * CHUNK_COLS; e.bias_off = I.layer * 32 * (int)sizeof(float);
    e.inv_L = Ly.inv_L; e.L_in = Ly.L_in; e.L_pool = Ly.L_pool; e.L_next = Ly.L_next;
    e.row0 = I.chunk * 128; e.out_ch = Ly.out_ch;
    e.save_a = SAVE ? SL.a_off[I.layer] : -1; e.save_bits = SAVE ? SL.bits_off[I.layer] : -1;
  }
  __syncthreads();

  if (warp == MMA_WARP) {
    // ===================================== MMA issuer =====================================
    // Items (layer, chunk) are issued in order; item i waits only for the epilogue items that produce the input rows it
    // reads (need), so a layer starts while the previous layer's last chunks are still in their epilogue.
    unsigned gpar = 0;
    for (int g = blockIdx.x; g < n_groups; g += gridDim.x, gpar ^= 1) {
      int waited = 0;   // done_bar[0 .. waited) observed in this group
      for (int it = 0; it < n_items; ++it) {
        const ItemDev I = S->item[it];
        for (; waited <= I.need; ++waited) mbar_wait(smem_addr(&S->done_bar[waited]), gpar);
        tc_fence_after();
        if (elect_one()) {
          if (I.first) {
            if (I.N == 64) issue_first<64, PASSES>(I.count, I.d, I.a_hi, I.b);
            else issue_first<32, PASSES>(I.count, I.d, I.a_hi, I.b);
          } else {
            issue_shifted<PASSES>(I.count, I.d, I.a_hi, I.a_lo, I.b);
          }
          mma_commit(smem_addr(&S->acc_bar[it]));
        }
        __syncwarp();
      }
    }
  } else {
    // ===================================== epilogue warps =====================================
    // every item is processed by all 16 warps: warp = (column quarter, lane quarter); a thread owns 8 channels of one row
    const int quarter = warp & 3, cq = warp >> 2;
    const int row_c = quarter * 32 + lane;     // row inside a chunk = TMEM lane
    const unsigned trow = tmem_base + ((unsigned)(quarter * 32) << 16) + cq * 8;
    const unsigned bias_base = smem_addr(bias_s) + cq * 8 * (int)sizeof(float);
    const Layer& L0y = TP.layer[0];
    const int rows0 = TP.n_chunks[0] * 128 < PLANE_ROWS ? TP.n_chunks[0] * 128 : PLANE_ROWS;
    const int rpw = (rows0 + EPI_WARPS - 1) / EPI_WARPS;            // im2col rows per warp
    const int r_lo = warp * rpw, r_hi = min(rows0, r_lo + rpw);
    const int planes0 = 2 * L0y.ksteps, taps0 = L0y.taps;
    // im2col scatter tasks of this lane: (row, input position, haplotype) -> one 1.0 of the one-hot row.  The mapping is
    // the same for every group; the codes of the NEXT group are fetched one group ahead and stay in registers.
    unsigned t_row[MAX_TASKS];   // shared address of the row (plane 0), 0 = no task
    int t_col[MAX_TASKS], t_var[MAX_TASKS], t_off[MAX_TASKS];
#pragma unroll
    for (int k = 0; k < MAX_TASKS; ++k) {
      const int task = lane + 32 * k;
      const int h = task & 1, rt = task >> 1;
      const int tt = rt % taps0, j = r_lo + rt / taps0;
      const int v = j / L0, pos = j - v * L0 + tt;
      const bool ok = j < r_hi && pos < L0;
      t_row[k] = ok ? act + j * 16 : 0u;
      t_col[k] = tt * C0 + h;
      t_var[k] = ok ? v : (1 << 30);
      t_off[k] = ok ? (int)(v * hap_stride) + h * L0 + pos : 0;
    }
    int codes[MAX_TASKS];
    auto fetch_codes = [&](int g) {
      const long long base = (long long)g * G * hap_stride;
      const int nv = g < n_groups ? min(G, n_variants - g * G) : 0;
      if (hap_kind == PMT_I64) {
#pragma unroll
        for (int k = 0; k < MAX_TASKS; ++k) codes[k] = t_var[k] < nv ? (int)__ldg(reinterpret_cast<const long long*>(haps) + base + t_off[k]) : -1;
      } else {
#pragma unroll
        for (int k = 0; k < MAX_TASKS; ++k) codes[k] = t_var[k] < nv ? (int)__ldg(reinterpret_cast<const short*>(haps) + base + t_off[k]) : -1;
      }
    };
    fetch_codes(blockIdx.x);
    unsigned gpar = 0;
    for (int g = blockIdx.x; g < n_groups; g += gridDim.x, gpar ^= 1) {
      const int v0 = g * G, nv = min(G, n_variants - v0);
      // ---- im2col rows of the first conv (batch.py:115-130): zero this warp's rows, then scatter the ones ----
      for (int j = r_lo + lane; j < r_hi; j += 32) {
        const unsigned ra = act + j * 16;
#pragma unroll
        for (int pl = 0; pl < 16; ++pl)
          if (pl < planes0) sts128(ra + pl * PLANE_BYTES, make_float4(0.f, 0.f, 0.f, 0.f));
      }
      __syncwarp();
#pragma unroll
      for (int k = 0; k < MAX_TASKS; ++k) {
        if ((unsigned)codes[k] < 5u) {
          const int col = t_col[k] + 2 * codes[k];
          sts_f32(t_row[k] + (col >> 2) * PLANE_BYTES + (col & 3) * 4, 1.f);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_addr(&S->done_bar[0]));
      fetch_codes(g + gridDim.x);

      for (int it = 0; it < n_items; ++it) {
        const unsigned ea = smem_addr(&S->epi[it]);
        const float4 e0f = lds128(ea), e1f = lds128(ea + 16), e2f = lds128(ea + 32);
        const int flags = __float_as_int(e0f.x), N = __float_as_int(e0f.y);
        const unsigned tcol = trow + __float_as_int(e0f.z);
        const unsigned bias_a = bias_base + __float_as_int(e0f.w);
        const int inv_L = __float_as_int(e1f.x), L_in = __float_as_int(e1f.y), L_pool = __float_as_int(e1f.z), L_next = __float_as_int(e1f.w);
        const int out_ch = __float_as_int(e2f.y);
        const int save_a = __float_as_int(e2f.z), save_bits = __float_as_int(e2f.w);
        unsigned win = 0;   // SAVE: bit i = the second element of the pooling window won for channel 8 cq + i
        const int j = __float_as_int(e2f.x) + row_c;
        const int v = (j * inv_L) >> 16, pos = j - v * L_in;
        int pp = pos;
        bool valid = v < nv;
        if (flags & F_POOL2) { valid = valid && !(pos & 1); pp = pos >> 1; }
        valid = valid && pp < L_pool;
        const float4 b0 = lds128(bias_a), b1 = lds128(bias_a + 16);
        mbar_wait(smem_addr(&S->acc_bar[it]), gpar);
        tc_fence_after();
        float x[8];
        {
          unsigned r[8], rl[8];
          tmem_ld8(tcol, r);
          if (PASSES == 3) tmem_ld8(tcol + N, rl);
          if (flags & F_DUP) {
            unsigned r2[8], rl2[8];
            tmem_ld8(tcol + 32, r2);
            if (PASSES == 3) tmem_ld8(tcol + N + 32, rl2);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float u0 = PASSES == 3 ? __uint_as_float(r[i]) + __uint_as_float(rl[i]) : __uint_as_float(r[i]);
              const float u1 = PASSES == 3 ? __uint_as_float(r2[i]) + __uint_as_float(rl2[i]) : __uint_as_float(r2[i]);
              x[i] = fmaxf(u0, u1);
              if (SAVE) win |= (u1 > u0 ? 1u : 0u) << i;
            }
          } else {
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = PASSES == 3 ? __uint_as_float(r[i]) + __uint_as_float(rl[i]) : __uint_as_float(r[i]);
          }
        }
        tc_fence_before();   // the accumulator has been read: a later item may overwrite it once this warp has arrived
        if (flags & F_POOL2) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float o = __shfl_xor_sync(0xffffffffu, x[i], 1);
            if (SAVE) win |= (o > x[i] ? 1u : 0u) << i;   // read on the even row of the pair: o is the odd row's value
            x[i] = fmaxf(x[i], o);
          }
        }
        x[0] += b0.x; x[1] += b0.y; x[2] += b0.z; x[3] += b0.w; x[4] += b1.x; x[5] += b1.y; x[6] += b1.z; x[7] += b1.w;
        if (flags & F_GLOBAL) {
          if (valid) {
            float* dst = info_seq + (long long)(v0 + v) * (D.d_info + D.d_seq) + D.d_info + cq * 8;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (cq * 8 + i < out_ch) dst[i] = (flags & F_SELU) ? SELU_SCALE * selu_u(x[i]) : x[i];
          }
        } else {
          if (flags & F_SELU) {
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = selu_u(x[i]);
          }
          if (SAVE && valid && save_a >= 0) {   // training: a_l (and the window bits) for the backward (pmt_cnn_bwd.cu)
            const int cols = G * L_next, col = v * L_next + pp;
            float* sg = save + (size_t)g * SL.group_floats;
            float* dstg = sg + save_a + (cq * 8) * cols + col;
#pragma unroll
            for (int i = 0; i < 8; ++i) dstg[i * cols] = rna_tf32(x[i]);   // rounded to TF32: the backward's MMAs read them as they lie
            if (save_bits >= 0) reinterpret_cast<unsigned char*>(sg + save_bits)[cq * cols + col] = (unsigned char)win;
          }
          if (!SAVE && (flags & F_TAIL)) {   // the split forward: fp32 into the tail kernel's A layout (pmt_cnn_tc.cuh)
            if (valid) {
              const int gv = v0 + v;
              float* dst = tail_buf + ((size_t)(gv >> 7) * (L_next * 8) + pp * 8 + 2 * cq) * (TAIL_PLANE / 4) + (gv & 127) * 4;
              *reinterpret_cast<float4*>(dst) = make_float4(x[0], x[1], x[2], x[3]);
              *reinterpret_cast<float4*>(dst + TAIL_PLANE / 4) = make_float4(x[4], x[5], x[6], x[7]);
            }
          } else if (valid) {
            const unsigned dst = act + (2 * cq) * PLANE_BYTES + (v * L_next + pp) * 16;
            sts128(dst, make_float4(x[0], x[1], x[2], x[3]));
            sts128(dst + PLANE_BYTES, make_float4(x[4], x[5], x[6], x[7]));
            if (PASSES == 3) {
#pragma unroll
              for (int i = 0; i < 8; ++i) x[i] -= __uint_as_float(__float_as_uint(x[i]) & 0xFFFFE000u);
              sts128(dst + BUF_BYTES, make_float4(x[0], x[1], x[2], x[3]));
              sts128(dst + BUF_BYTES + PLANE_BYTES, make_float4(x[4], x[5], x[6], x[7]));
            }
          }
          fence_proxy_async();
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_addr(&S->done_bar[1 + it]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc<CNN_TMEM_COLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// The tail of the split forward (pmt_cnn_tc.cuh: TailPlan): persistent CTAs over tiles of 128 variants, M = 128.
//   warps 0-7  epilogue: thread = variant (TMEM lane) x 16 output channels; they also derive each stage's A_lo rows from
//              the A_hi rows the loader brought in (A_hi is the fp32 activation itself: the MMA reads its TF32 part).
//   warp  8    MMA issuer: the first tail layer streams its K through TAIL_STAGES stages of 32 floats, the others read
//              the previous tail layer's output from the `mid` buffer.
//   warp  9    loader: one bulk copy per stage.
// TMEM: the first layer's accumulator in columns [0, 2 N0), tail layer t >= 1 (N = 32) in [64 + 64 t, 128 + 64 t).
// Every wait's phase follows from the stage-use counter u or the tile counter it.
// ------------------------------------------------------------------------------------------------
struct TailBars {
  unsigned long long loaded[TAIL_STAGES];   // A_hi of the stage landed (expect_tx)
  unsigned long long full[TAIL_STAGES];     // A_lo written (epilogue warps)
  unsigned long long empty[TAIL_STAGES];    // the stage's MMAs completed (tcgen05.commit)
  unsigned long long acc[MAX_TAIL];         // tail layer t's accumulator complete
  unsigned long long mid;                   // the mid buffer holds the next tail layer's input (epilogue warps)
  unsigned long long free0;                 // the first layer's accumulator has been read (epilogue warps)
  unsigned tmem_base;
  int pad_;
};
constexpr int TAIL_TMEM_COLS = 256;
__host__ __device__ constexpr int tail_acc_col(int t) { return t == 0 ? 0 : 64 + 64 * t; }

// 4 k-steps of one dense tail layer: A (128 rows) and B in the no-swizzle K-major layout, K chunks TAIL_PLANE apart in A
template <int N, int PASSES>
__device__ __forceinline__ void issue_dense(unsigned d, unsigned a_hi, unsigned a_lo, unsigned b, bool first) {
  constexpr int R = 2 * N;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    const unsigned ao = (unsigned)(2 * ks * (TAIL_PLANE / 16)), bo = (unsigned)(2 * ks * R);
    const unsigned acc = (first && ks == 0) ? 0u : 1u;
    if (PASSES == 3) {
      mma_ss_desc_lo<make_idesc(2 * N)>(d, a_hi + ao, b + bo, acc);
      mma_ss_desc_lo<make_idesc(N)>(d, a_lo + ao, b + bo, 1u);
    } else {
      mma_ss_desc_lo<make_idesc(N)>(d, a_hi + ao, b + bo, acc);
    }
  }
}
template <int PASSES>
__device__ __forceinline__ void issue_dense_n(int N, unsigned d, unsigned a_hi, unsigned a_lo, unsigned b, bool first) {
  if (N == 64) issue_dense<64, PASSES>(d, a_hi, a_lo, b, first);
  else issue_dense<32, PASSES>(d, a_hi, a_lo, b, first);
}

template <int PASSES>
__global__ void __launch_bounds__(TAIL_THREADS, 1)
hap_cnn_tail_kernel(const __grid_constant__ TailPlan TT, const unsigned char* __restrict__ image, const float* __restrict__ wflat,
                    const __grid_constant__ PmtModelDesc D, const float* __restrict__ tail_buf, int n_variants,
                    float* __restrict__ info_seq) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* p = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const unsigned stage_s = smem_addr(p); p += TAIL_STAGES * 2 * TAIL_STAGE_BYTES;   // stage s: A_hi, then A_lo
  const unsigned mid_s = smem_addr(p); p += 2 * TAIL_STAGE_BYTES;                    // A_hi, A_lo of tail layers 1..
  unsigned char* img_s = p; p += TT.image_bytes;
  float* bias_s = reinterpret_cast<float*>(p); p += MAX_TAIL * 32 * sizeof(float);
  TailBars* S = reinterpret_cast<TailBars*>((reinterpret_cast<uintptr_t>(p) + 15) & ~uintptr_t(15));

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int lane = tid & 31;
  const int nt = TT.n_layers, ns = TT.K0 / (4 * TAIL_STAGE_CHUNKS);   // stages per tile
  const int n_tiles = (n_variants + 127) / 128;

  if (tid == 0) {
    for (int s = 0; s < TAIL_STAGES; ++s) {
      mbar_init(smem_addr(&S->loaded[s]), 1);
      mbar_init(smem_addr(&S->full[s]), TAIL_EPI_WARPS);
      mbar_init(smem_addr(&S->empty[s]), 1);
    }
    for (int t = 0; t < MAX_TAIL; ++t) mbar_init(smem_addr(&S->acc[t]), 1);
    mbar_init(smem_addr(&S->mid), TAIL_EPI_WARPS);
    mbar_init(smem_addr(&S->free0), TAIL_EPI_WARPS);
    fence_mbar_init();
  }
  for (int i = tid; i < TT.image_bytes / 16; i += TAIL_THREADS)
    reinterpret_cast<uint4*>(img_s)[i] = __ldg(reinterpret_cast<const uint4*>(image) + i);
  for (int i = tid; i < nt * 32; i += TAIL_THREADS) {
    const Layer& Ly = TT.layer[i / 32];
    const int n = i % 32, b_off = D.cnn_ops[Ly.op].b_off;
    bias_s[i] = (n < Ly.out_ch && b_off >= 0) ? __ldg(wflat + b_off + n) : 0.f;
  }
  if (warp == TAIL_EPI_WARPS) tmem_alloc<TAIL_TMEM_COLS>(smem_addr(&S->tmem_base));
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = __shfl_sync(0xffffffffu, S->tmem_base, 0);
  const unsigned img_a = smem_addr(img_s);

  if (warp == TAIL_EPI_WARPS + 1) {
    // ===================================== loader =====================================
    if (elect_one()) {
      int u = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const float* src = tail_buf + (size_t)tile * (TT.K0 / 4) * (TAIL_PLANE / 4);
        for (int k = 0; k < ns; ++k, ++u) {
          const int s = u % TAIL_STAGES;
          if (u >= TAIL_STAGES) mbar_wait(smem_addr(&S->empty[s]), (u / TAIL_STAGES - 1) & 1);
          mbar_expect_tx(smem_addr(&S->loaded[s]), TAIL_STAGE_BYTES);
          bulk_g2s(stage_s + s * 2 * TAIL_STAGE_BYTES, src + (size_t)k * (TAIL_STAGE_BYTES / 4), TAIL_STAGE_BYTES,
                   smem_addr(&S->loaded[s]));
        }
      }
    }
    __syncwarp();
  } else if (warp == TAIL_EPI_WARPS) {
    // ===================================== MMA issuer =====================================
    const Layer& L0y = TT.layer[0];
    const int N0 = L0y.N;
    int u = 0;
    for (int tile = blockIdx.x, it = 0; tile < n_tiles; tile += gridDim.x, ++it) {
      if (it > 0) mbar_wait(smem_addr(&S->free0), (it - 1) & 1);
      for (int k = 0; k < ns; ++k, ++u) {
        const int s = u % TAIL_STAGES;
        mbar_wait(smem_addr(&S->full[s]), (u / TAIL_STAGES) & 1);
        tc_fence_after();
        if (elect_one()) {
          const unsigned a = stage_s + s * 2 * TAIL_STAGE_BYTES;
          const unsigned b = img_a + L0y.img_off + k * TAIL_STAGE_CHUNKS * (2 * N0 * 16);
          issue_dense_n<PASSES>(N0, tmem_base, desc_lo(a, TAIL_PLANE), desc_lo(a + TAIL_STAGE_BYTES, TAIL_PLANE), desc_lo(b, 2 * N0 * 16),
                                k == 0);
          mma_commit(smem_addr(&S->empty[s]));
          if (k == ns - 1) mma_commit(smem_addr(&S->acc[0]));
        }
        __syncwarp();
      }
      for (int t = 1; t < nt; ++t) {
        const Layer& Ly = TT.layer[t];
        mbar_wait(smem_addr(&S->mid), (it * (nt - 1) + t - 1) & 1);
        tc_fence_after();
        if (elect_one()) {
          issue_dense_n<PASSES>(Ly.N, tmem_base + tail_acc_col(t), desc_lo(mid_s, TAIL_PLANE), desc_lo(mid_s + TAIL_STAGE_BYTES, TAIL_PLANE),
                                desc_lo(img_a + Ly.img_off, 2 * Ly.N * 16), true);
          mma_commit(smem_addr(&S->acc[t]));
        }
        __syncwarp();
      }
    }
  } else {
    // ===================================== epilogue warps =====================================
    const int quarter = warp & 3, cq = warp >> 2;
    const int row = quarter * 32 + lane;       // TMEM lane = variant inside the tile
    const int c0 = cq * 16;                    // this thread's 16 output channels
    const unsigned trow = tmem_base + ((unsigned)(quarter * 32) << 16) + c0;
    int u = 0;
    for (int tile = blockIdx.x, it = 0; tile < n_tiles; tile += gridDim.x, ++it) {
      for (int k = 0; k < ns; ++k, ++u) {
        const int s = u % TAIL_STAGES;
        mbar_wait(smem_addr(&S->loaded[s]), (u / TAIL_STAGES) & 1);
        if (PASSES == 3) {   // A_lo = A - its TF32 part, as the head layers' epilogue splits its activations
          const unsigned hi = stage_s + s * 2 * TAIL_STAGE_BYTES;
#pragma unroll
          for (int i = 0; i < TAIL_STAGE_BYTES / 16 / (32 * TAIL_EPI_WARPS); ++i) {
            const unsigned o = (unsigned)((i * 32 * TAIL_EPI_WARPS + tid) * 16);
            float4 v = lds128(hi + o);
            v.x -= __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
            v.y -= __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
            v.z -= __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
            v.w -= __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
            sts128(hi + TAIL_STAGE_BYTES + o, v);
          }
          fence_proxy_async();
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_addr(&S->full[s]));
      }
      const int gv = tile * 128 + row;
      const bool valid = gv < n_variants;
      for (int t = 0; t < nt; ++t) {
        const Layer& Ly = TT.layer[t];
        const int N = Ly.N;
        const unsigned tcol = trow + tail_acc_col(t);
        const unsigned bias_a = smem_addr(bias_s) + (t * 32 + c0) * (int)sizeof(float);
        mbar_wait(smem_addr(&S->acc[t]), it & 1);
        tc_fence_after();
        float x[16];
        {
          unsigned r[16], rl[16];
          tmem_ld16(tcol, r);
          if (PASSES == 3) tmem_ld16(tcol + N, rl);
          if (Ly.pool2) {   // N = 64: the conv at the two positions of the pooling window, side by side
            unsigned r2[16], rl2[16];
            tmem_ld16(tcol + 32, r2);
            if (PASSES == 3) tmem_ld16(tcol + N + 32, rl2);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float u0 = PASSES == 3 ? __uint_as_float(r[i]) + __uint_as_float(rl[i]) : __uint_as_float(r[i]);
              const float u1 = PASSES == 3 ? __uint_as_float(r2[i]) + __uint_as_float(rl2[i]) : __uint_as_float(r2[i]);
              x[i] = fmaxf(u0, u1);
            }
          } else {
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) x[i] = PASSES == 3 ? __uint_as_float(r[i]) + __uint_as_float(rl[i]) : __uint_as_float(r[i]);
          }
        }
        tc_fence_before();   // the accumulator has been read
        if (t == 0) {
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_addr(&S->free0));
        }
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
          const float4 b = lds128(bias_a + i * 4);
          x[i] += b.x; x[i + 1] += b.y; x[i + 2] += b.z; x[i + 3] += b.w;
        }
        const bool selu = Ly.act == PMT_ACT_SELU;
        if (Ly.to_global) {
          if (valid) {
            float* dst = info_seq + (long long)gv * (D.d_info + D.d_seq) + D.d_info + c0;
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (c0 + i < Ly.out_ch) dst[i] = selu ? SELU_SCALE * selu_u(x[i]) : x[i];
          }
        } else {
          if (selu) selu_u_n<16>(x);
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const unsigned dst = mid_s + ((c0 + i) / 4) * TAIL_PLANE + row * 16;
            sts128(dst, make_float4(x[i], x[i + 1], x[i + 2], x[i + 3]));
            if (PASSES == 3) {
#pragma unroll
              for (int j = i; j < i + 4; ++j) x[j] -= __uint_as_float(__float_as_uint(x[j]) & 0xFFFFE000u);
              sts128(dst + TAIL_STAGE_BYTES, make_float4(x[i], x[i + 1], x[i + 2], x[i + 3]));
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_addr(&S->mid));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == TAIL_EPI_WARPS) tmem_dealloc<TAIL_TMEM_COLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// Weight images, B operand in the no-swizzle K-major layout [tap][16-byte K chunk][row][4 floats]; a plane holds
// 2N rows: rows [0, N) = TF32-rounded W, rows [N, 2N) = the remainder W - W_hi.
// ------------------------------------------------------------------------------------------------
__device__ float cnn_weight(const PmtModelDesc& D, const Layer& Ly, const float* __restrict__ w, int tap, int n, int k) {
  const PmtCnnOp& op = D.cnn_ops[Ly.op];
  if (Ly.first) {   // k = tt * C0 + ch over the im2col row; columns [32, 64) are the conv one position later
    const int tt = k / C0, ch = k - tt * C0;
    const int co = n & 31, t = tt - (n >> 5);
    if (co >= op.out_ch || t < 0 || t >= op.ksize || tt >= Ly.taps) return 0.f;
    return w[op.w_off + (co * op.in_ch + ch) * op.ksize + t];
  }
  if (n >= op.out_ch || k >= Ly.in_ch) return 0.f;
  const float s = Ly.scale_in ? SELU_SCALE : 1.f;
  if (Ly.is_linear) return s * w[op.w_off + n * op.in_ch + (Ly.flat_len > 1 ? k * Ly.flat_len + tap : k)];   // flatten is channel-major
  return s * w[op.w_off + (n * op.in_ch + k) * op.ksize + tap];
}

__global__ void pack_cnn_tc_kernel(const __grid_constant__ PmtModelDesc D, const __grid_constant__ Plan TP, const float* __restrict__ w,
                                   unsigned char* __restrict__ image) {
  const Layer& Ly = TP.layer[blockIdx.x];
  const int N = Ly.N, R = 2 * N;
  const int taps = Ly.first ? 1 : Ly.taps, chunks = Ly.first ? 2 * Ly.ksteps : 8;
  for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < taps * chunks * R * 4; idx += gridDim.y * blockDim.x) {
    const int e = idx & 3, r = (idx >> 2) % R, ch = (idx >> 2) / R % chunks, tap = (idx >> 2) / R / chunks;
    const float v = cnn_weight(D, Ly, w, tap, r % N, ch * 4 + e);
    const float hi = rna_tf32(v);
    *reinterpret_cast<float*>(image + (size_t)Ly.img_off + (size_t)idx * 4) = r < N ? hi : v - hi;
  }
}

// tail images: a dense layer over the whole input window.  Row n = 32 pos + co (hi rows [0, N), remainders [N, 2N)) holds
// output position pos; K column kk = 32 p + ci is input position p, channel ci: the conv's tap p - pos
__global__ void pack_cnn_tail_kernel(const __grid_constant__ PmtModelDesc D, const __grid_constant__ TailPlan TT, const float* __restrict__ w,
                                     unsigned char* __restrict__ image) {
  const Layer& Ly = TT.layer[blockIdx.x];
  const int N = Ly.N, R = 2 * N, chunks = Ly.L_in * 8;
  for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < chunks * R * 4; idx += gridDim.y * blockDim.x) {
    const int e = idx & 3, r = (idx >> 2) % R, ch = (idx >> 2) / R;
    const int kk = ch * 4 + e, n = r % N, tap = (kk >> 5) - (n >> 5);
    const float v = tap >= 0 && tap < Ly.taps ? cnn_weight(D, Ly, w, tap, n & 31, kk & 31) : 0.f;
    const float hi = rna_tf32(v);
    *reinterpret_cast<float*>(image + (size_t)Ly.img_off + (size_t)idx * 4) = r < N ? hi : v - hi;
  }
}

}  // namespace cnntc
}  // namespace pmt

// ================================================================================================
// host side
// ================================================================================================
using namespace pmt;
using namespace pmt::cnntc;

static bool schedule_groups(cnntc::Plan& T, int hap_len);

// Builds the layer program; returns false when the CNN is outside this kernel's envelope (the FP32 SIMT kernel
// hap_cnn_kernel then runs instead).
bool pmt_build_cnn_tc_plan(const pmt::Plan& P, cnntc::Plan* out) {
  cnntc::Plan& T = *out;
  memset(&T, 0, sizeof(T));
  const PmtModelDesc& d = P.d;
  T.L0 = d.hap_len;
  if (d.n_cnn_ops < 2 || d.hap_len < 1 || d.d_seq > 32) return false;
  int i = 0, L = d.hap_len, ch = C0;
  bool prev_selu = false;
  while (i < d.n_cnn_ops) {
    const PmtCnnOp& op = d.cnn_ops[i];
    if (T.n_layers >= MAX_LAYERS) return false;
    Layer& Ly = T.layer[T.n_layers];
    memset(&Ly, 0, sizeof(Ly));
    Ly.op = i;
    Ly.act = op.act;
    if (op.act != PMT_ACT_NONE && op.act != PMT_ACT_SELU) return false;
    if (op.kind == PMT_CNN_CONV) {
      if (op.stride != 1 || op.in_ch != ch || op.out_ch > 32 || op.in_len != L || op.ksize < 1 || op.ksize > 8 || op.out_len != L - op.ksize + 1 ||
          op.out_len < 1)
        return false;
      Ly.first = T.n_layers == 0;
      if (!Ly.first && op.in_ch > 32) return false;
      Ly.L_in = L; Ly.L_out = op.out_len; Ly.L_pool = op.out_len;
      Ly.ksize = op.ksize; Ly.in_ch = op.in_ch; Ly.out_ch = op.out_ch; Ly.scale_in = prev_selu;
      // pools that follow (a monotone activation commutes with max-pooling and was folded into the conv's act)
      int j = i + 1;
      for (; j < d.n_cnn_ops && d.cnn_ops[j].kind == PMT_CNN_POOL; ++j) {
        const PmtCnnOp& pl = d.cnn_ops[j];
        if (pl.ksize == 1 && pl.stride == 1) continue;
        if (Ly.dup || Ly.pool2 || pl.ksize != 2) return false;
        if (pl.stride == 1 && Ly.first) { Ly.dup = 1; Ly.L_pool = Ly.L_out - 1; }
        else if (pl.stride == 2 && (L % 2 == 0)) { Ly.pool2 = 1; Ly.L_pool = Ly.L_out / 2; }
        else return false;
        if (pl.out_len != Ly.L_pool || Ly.L_pool < 1) return false;
      }
      Ly.taps = Ly.first ? op.ksize + Ly.dup : op.ksize;
      if (Ly.first) {
        Ly.ksteps = (Ly.taps * C0 + 7) / 8;
        if (Ly.ksteps > 8) return false;
        Ly.N = Ly.dup ? 64 : 32;
      } else {
        Ly.N = 32;
      }
      Ly.L_next = Ly.L_pool;
      L = Ly.L_pool; ch = op.out_ch;
      prev_selu = op.act == PMT_ACT_SELU;
      i = j;
    } else if (op.kind == PMT_CNN_LINEAR) {
      if (T.n_layers == 0 || op.out_ch > 32) return false;
      Ly.is_linear = 1;
      Ly.flat_len = L;                       // first linear consumes the flattened [ch][L] map as a conv of kernel L
      if (L > 8 || op.in_ch != ch * L || ch > 32) return false;
      Ly.taps = L; Ly.ksize = L; Ly.in_ch = ch; Ly.out_ch = op.out_ch; Ly.scale_in = prev_selu;
      Ly.L_in = L; Ly.L_out = 1; Ly.L_pool = 1; Ly.L_next = 1; Ly.N = 32;
      L = 1; ch = op.out_ch;
      prev_selu = op.act == PMT_ACT_SELU;
      ++i;
    } else {
      return false;   // a pool before any conv
    }
    ++T.n_layers;
  }
  if (T.n_layers < 2 || !T.layer[T.n_layers - 1].is_linear || T.layer[T.n_layers - 1].out_ch != d.d_seq) return false;
  T.layer[T.n_layers - 1].to_global = 1;
  // images
  int bytes = 0;
  for (int l = 0; l < T.n_layers; ++l) {
    Layer& Ly = T.layer[l];
    Ly.img_off = bytes;
    Ly.img_bytes = (Ly.first ? 2 * Ly.ksteps : Ly.taps * 8) * 2 * Ly.N * 16;   // hi and lo rows interleaved per plane
    bytes += Ly.img_bytes;
    Ly.inv_L = 65536 / Ly.L_in + 1;
  }
  T.image_bytes = bytes;
  return schedule_groups(T, d.hap_len);
}

// The group size G and the item list of hap_cnn_tc_kernel over T's layers.
static bool schedule_groups(cnntc::Plan& T, int hap_len) {
  const int bytes = T.image_bytes;
  // variants per group: every layer's rows must fit MAX_CHUNKS chunks and the planes; pick the G with the fewest MMA
  // cycles per variant
  // Every layer's weight image stays resident in shared memory next to the two activation buffers: that is the kernel's
  // capacity limit.  v0.4.0's layer strings on haplotypes of 21 bases fit with 4.4 KB to spare; on 25 bases they leave
  // 2 positions to the flatten, whose 2-tap Linear image (16 KB instead of 8 KB) is 3.6 KB too many, and that shape runs
  // on the FP32 SIMT kernel (hap_cnn_kernel).
  const int fixed = 2 * BUF_BYTES + bytes + MAX_LAYERS * 32 * 4 + (int)sizeof(Bars) + 1024 + 64;
  if (fixed > 227 * 1024) return false;
  T.smem = fixed;
  double best = 1e30;
  int best_g = 0;
  for (int G = 1; G <= 128; ++G) {
    if (G * hap_len > PLANE_ROWS) break;
    double cost = 0;
    bool ok = true;
    for (int l = 0; l < T.n_layers; ++l) {
      const Layer& Ly = T.layer[l];
      const int chunks = (G * Ly.L_in + 127) / 128;
      if (chunks > MAX_CHUNKS) ok = false;
      cost += chunks * (Ly.first ? Ly.ksteps : Ly.taps * 4) * (Ly.N / 2) + 600.0;   // + per-layer hand-off
    }
    if (ok && cost / G < best) { best = cost / G; best_g = G; }
  }
  if (best_g == 0) return false;
  T.G = best_g;
  for (int l = 0; l < T.n_layers; ++l) T.n_chunks[l] = (T.G * T.layer[l].L_in + 127) / 128;
  {   // the im2col scatter keeps its one-hot entries in MAX_TASKS registers per lane
    const int rows0 = T.n_chunks[0] * 128 < PLANE_ROWS ? T.n_chunks[0] * 128 : PLANE_ROWS;
    const int rpw = (rows0 + EPI_WARPS - 1) / EPI_WARPS;
    if ((rpw * T.layer[0].taps * 2 + 31) / 32 > MAX_TASKS) return false;
  }
  // work items in issue order, with the epilogue item each one depends on
  int first_item[MAX_LAYERS];
  for (int l = 0; l < T.n_layers; ++l) {
    first_item[l] = T.n_items;
    const Layer& Ly = T.layer[l];
    for (int c = 0; c < T.n_chunks[l]; ++c) {
      if (T.n_items >= MAX_ITEMS) return false;
      Item& I = T.item[T.n_items];
      I.layer = l; I.chunk = c; I.need = 0;
      if (l > 0) {
        const Layer& Pv = T.layer[l - 1];
        const int taps = Ly.taps, s = Pv.pool2 ? 2 : 1;
        int last_row = 128 * c + 128 + taps - 2;                    // last input row the chunk's MMAs read
        if (last_row > T.G * Ly.L_in - 1) last_row = T.G * Ly.L_in - 1;
        const int v = last_row / Ly.L_in, pq = last_row % Ly.L_in;  // written by the previous layer's row (v, pq * s)
        int src_chunk = (v * Pv.L_in + pq * s) / 128;
        if (src_chunk < c && c < T.n_chunks[l - 1]) src_chunk = c;   // the accumulator columns of (l-1, c) are reused
        if (src_chunk > T.n_chunks[l - 1] - 1) src_chunk = T.n_chunks[l - 1] - 1;
        I.need = 1 + first_item[l - 1] + src_chunk;
        if (T.n_items > 0 && I.need < T.item[T.n_items - 1].need) I.need = T.item[T.n_items - 1].need;
      }
      ++T.n_items;
    }
  }
  return true;
}

bool pmt_build_cnn_split_plan(const cnntc::Plan& T, int hap_len, cnntc::Plan* head, cnntc::TailPlan* tail) {
  cnntc::Plan& H = *head;
  cnntc::TailPlan& TT = *tail;
  memset(&H, 0, sizeof(H));
  memset(&TT, 0, sizeof(TT));
  int s = -1;   // the first tail layer: the earliest from which every layer qualifies
  for (int c = 1; c < T.n_layers && s < 0; ++c) {
    bool ok = T.n_layers - c <= MAX_TAIL;
    for (int l = c; ok && l < T.n_layers; ++l) {
      const Layer& Ly = T.layer[l];
      ok = Ly.L_pool == 1 && (Ly.L_out == 1 || (Ly.L_out == 2 && Ly.pool2)) && Ly.L_in * 32 <= (l == c ? TAIL_MAX_K : 32);
    }
    if (ok) s = c;
  }
  if (s < 0) return false;
  TT.n_layers = T.n_layers - s;
  TT.K0 = T.layer[s].L_in * 32;
  TT.image_off = (T.image_bytes + 255) & ~255;
  int bytes = 0;
  for (int t = 0; t < TT.n_layers; ++t) {
    Layer& Ly = TT.layer[t];
    Ly = T.layer[s + t];
    Ly.N = 32 * Ly.L_out;
    Ly.img_off = bytes;
    Ly.img_bytes = Ly.L_in * 8 * 2 * Ly.N * 16;
    bytes += Ly.img_bytes;
  }
  TT.image_bytes = bytes;
  TT.smem = 1024 + TAIL_STAGES * 2 * TAIL_STAGE_BYTES + 2 * TAIL_STAGE_BYTES + bytes + MAX_TAIL * 32 * 4 + (int)sizeof(TailBars) + 64;
  if (TT.smem > 227 * 1024) return false;
  // the head: the layers before s, their images where the single kernel has them
  H.n_layers = s;
  H.L0 = T.L0;
  for (int l = 0; l < s; ++l) H.layer[l] = T.layer[l];
  H.layer[s - 1].to_tail = 1;
  H.image_bytes = T.layer[s].img_off;
  return schedule_groups(H, hap_len);
}

size_t pmt_cnn_tc_image_bytes(const CallPlan& C) {
  if (!C.cnn_tc_ok) return 0;
  return (C.cnn_split ? (size_t)C.CT.image_off + C.CT.image_bytes : (size_t)C.C.image_bytes) + 256;
}

template <int PASSES, bool SAVE>
static int launch_cnn_tc(const cnntc::Plan& T, const unsigned char* image, const float* weights, const PmtModelDesc& D, const void* haps,
                         const PmtBatch* batch, int n, float* info_seq, const SaveLayout& SL, float* save, int grid, cudaStream_t st,
                         float* tail_buf = nullptr) {
  PMT_CUDA(cudaFuncSetAttribute(hap_cnn_tc_kernel<PASSES, SAVE>, cudaFuncAttributeMaxDynamicSharedMemorySize, T.smem));
  hap_cnn_tc_kernel<PASSES, SAVE><<<grid, cnntc::THREADS, T.smem, st>>>(T, image, weights, D, haps, batch->hap_kind, batch->hap_stride, n, info_seq,
                                                               SL, save, tail_buf);
  return 0;
}

void pmt_cnn_save_layout(const cnntc::Plan& T, SaveLayout* out) {
  SaveLayout& S = *out;
  memset(&S, 0, sizeof(S));
  S.G = T.G; S.n_layers = T.n_layers;
  int off = 0;
  for (int l = 0; l < MAX_LAYERS; ++l) { S.a_off[l] = -1; S.bits_off[l] = -1; }
  for (int l = 0; l < T.n_layers; ++l) {
    const Layer& Ly = T.layer[l];
    if (Ly.to_global) continue;
    const int cols = T.G * Ly.L_next;
    S.a_off[l] = off; off += 32 * cols;
    if (Ly.dup || Ly.pool2) { S.bits_off[l] = off; off += cols; }   // [4][cols] bytes
  }
  S.group_floats = (off + 3) & ~3;
}

// Training recompute: always the split-precision mode (the saved activations are the fp32-parity ones).
int pmt_launch_cnn_tc_save(const pmt::Plan& P, const cnntc::Plan& T, const float* weights, const PmtBatch* batch, int v_first, int n,
                           float* info_seq, const unsigned char* image, float* save, int n_sm, cudaStream_t st) {
  SaveLayout SL;
  pmt_cnn_save_layout(T, &SL);
  const int n_groups = (n + T.G - 1) / T.G;
  const int grid = n_groups < n_sm ? n_groups : n_sm;
  const size_t esz = batch->hap_kind == PMT_I64 ? 8 : 2;
  const void* haps = reinterpret_cast<const unsigned char*>(batch->haplotypes) + (size_t)v_first * batch->hap_stride * esz;
  float* out = info_seq + (size_t)v_first * (P.d.d_info + P.d.d_seq);
  return launch_cnn_tc<3, true>(T, image, weights, P.d, haps, batch, n, out, SL, save, grid, st);
}

int pmt_pack_cnn_tc_images(const pmt::Plan& P, const cnntc::Plan& T, const float* weights, unsigned char* image, cudaStream_t st) {
  pack_cnn_tc_kernel<<<dim3(T.n_layers, 16), 256, 0, st>>>(P.d, T, weights, image);
  return 0;
}

template <int PASSES>
static int launch_cnn_tail(const TailPlan& TT, const unsigned char* image, const float* weights, const PmtModelDesc& D, const float* tail_buf,
                           int n, float* info_seq, int n_sm, cudaStream_t st) {
  const int n_tiles = (n + 127) / 128;
  PMT_CUDA(cudaFuncSetAttribute(hap_cnn_tail_kernel<PASSES>, cudaFuncAttributeMaxDynamicSharedMemorySize, TT.smem));
  hap_cnn_tail_kernel<PASSES><<<n_tiles < n_sm ? n_tiles : n_sm, TAIL_THREADS, TT.smem, st>>>(TT, image + TT.image_off, weights, D, tail_buf, n,
                                                                                               info_seq);
  return 0;
}

// W.cnn_tc_image: the weight images (16-byte aligned); W.cnn_tail: the head kernel's output to the tail kernel
int pmt_launch_cnn_tc(const CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq, const FwdBuffers& W,
                      bool reuse_image, cudaStream_t st) {
  unsigned char* image = W.cnn_tc_image;
  float* tail_buf = W.cnn_tail;
  if (!reuse_image) {   // both forms' images, so that a prepared call finds whichever it runs
    pack_cnn_tc_kernel<<<dim3(C.C.n_layers, 16), 256, 0, st>>>(C.P.d, C.C, weights, image);
    if (C.cnn_split) pack_cnn_tail_kernel<<<dim3(C.CT.n_layers, 16), 256, 0, st>>>(C.P.d, C.CT, weights, image + C.CT.image_off);
  }
  const bool split = C.cnn == CnnKernel::TC_TAIL;
  const cnntc::Plan& T = split ? C.CH : C.C;
  const int n = batch->n_variants;
  const int n_groups = (n + T.G - 1) / T.G;
  const int grid = n_groups < C.n_sm ? n_groups : C.n_sm;
  SaveLayout SL;
  memset(&SL, 0, sizeof(SL));
  if (C.passes == 1) {
    if (launch_cnn_tc<1, false>(T, image, weights, C.P.d, batch->haplotypes, batch, n, info_seq, SL, nullptr, grid, st, tail_buf)) return 1;
    return split ? launch_cnn_tail<1>(C.CT, image, weights, C.P.d, tail_buf, n, info_seq, C.n_sm, st) : 0;
  }
  if (launch_cnn_tc<3, false>(T, image, weights, C.P.d, batch->haplotypes, batch, n, info_seq, SL, nullptr, grid, st, tail_buf)) return 1;
  return split ? launch_cnn_tail<3>(C.CT, image, weights, C.P.d, tail_buf, n, info_seq, C.n_sm, st) : 0;
}
