// Tensor-core (tcgen05 / TMEM) backward of the read path for sm_100a: autograd of artifact_model.py:243-297 over the
// tile-sized read sets (misc_utils.py:125-127 calls loss.backward() through exactly these layers).
//
// Two kernels per range of tiles:
//   reads_forward_tc_kernel<3, SAVE>     (pmt_tc.cu) recomputes the forward and leaves every layer's operand in global
//       memory as PANELS (pmt_tc.cuh): the layout an MN-major tf32 operand of tcgen05.mma must have
//   reads_backward_tc_kernel             walks the layers in reverse.  Same organisation as the forward: one persistent
//       CTA per SM, two tiles of 128 reads in flight, 16 epilogue warps (two threads per read), one MMA-issuer warp per
//       slot, one loader warp.  Per layer and tile two MMA groups:
//         data gradient    dA[128 x K] = dY[128 x N] . W[N x K]   TS form: dY sits in TMEM (lane = read), the
//                          transposed, pre-swizzled weight image streams through a shared-memory ring
//         weight gradient  dW[K x N] = A^T[K x 128] . dY[128 x N]  SS form, BOTH operands MN-major: the reduction
//                          runs over the tile's reads, so the saved operand panel (bulk-copied from global memory) and the
//                          dY panel the epilogue wrote are consumed as they lie; 16 MMAs of 8 reads each
//       dW lands in TMEM (lane = input feature, column = output feature) and is flushed per tile with red.global.add
//       into a gradient buffer PRIVATE to the (CTA, slot) pair, in the layout of the folded weight images; biases are
//       the row of the constant-1 operand column.  unfold_kernel sums the private buffers in a fixed order and maps
//       the image gradients back through the folds of pack_tc_kernel (skip alpha, SELU scale, LayerNorm affine,
//       rotation + translation).  Tiles come from a deterministic tile list and go to slots statically, so every sum
//       has a fixed order: gradients are bitwise reproducible.
//   Per-row parameter gradients that are not GEMMs (gate scalars, SGU LayerNorm, regulariser, clustering head) are
//   reduced with warp shuffles into per-warp slots of the same private buffer.
// TMEM per slot (256 columns): G = dL/d(residual stream) (64), D = data-gradient accumulator (64), dY operand (64),
// dW accumulator (64).  Arithmetic: TF32 operands rounded to nearest, fp32 accumulation.
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "pmt_call.h"

namespace pmt {
namespace tc {

constexpr int COL_G = 0, COL_D = 64, COL_DY = 128, COL_DW = 192;
constexpr int OPBUF_BYTES = 4 * PANEL_BYTES;   // per slot: operand panels 0, 1, then dY panels 0, 1
constexpr int BW_TAB = 2 * BWD_MAXV * MAXH;    // floats of one per-variant table
constexpr int BXCH_ROWS = 16;                  // exchange buffer rows: hidden units, final features, 16 stream columns
constexpr int HEAD_K_STRIDE = MAXE + 5;        // per-cluster head gradient slots: unit[MAXE], tau, mu, emg sigma, lambda, log weight

struct SharedB {
  unsigned long long bar_a[2], bar_d[2], bar_w[2], act_full[2], act_free[2], wfull[NS_MAX], wfree[NS_MAX];
  unsigned tmem_base;
  int pad_;
  SlotMeta slot[2];
};

__device__ __forceinline__ float du(float a) { return a > 0.f ? 1.f : a + SELU_ALPHA; }   // u'(x) from a = u(x)

template <int NC>
__device__ __forceinline__ void load_act(unsigned act_s, int row, int col0, float* a) {
#pragma unroll
  for (int i = 0; i < NC / 4; ++i) {
    const float4 q = lds128(act_s + panel_off(row, col0 / 4 + i));
    a[4 * i] = q.x; a[4 * i + 1] = q.y; a[4 * i + 2] = q.z; a[4 * i + 3] = q.w;
  }
}
// dY columns [col0, col0 + NC) of this row (already rounded to TF32): TMEM operand of the data gradient and panel of the
// weight gradient
template <int NC>
__device__ __forceinline__ void store_dy(unsigned t_dy, unsigned dy_s, int row, int col0, const float* v) {
  unsigned r[NC];
#pragma unroll
  for (int i = 0; i < NC; ++i) r[i] = __float_as_uint(v[i]);
  if constexpr (NC == 24) { tmem_st16(t_dy + col0, r); tmem_st8(t_dy + col0 + 16, r + 16); }
  else tmem_st_n<NC>(t_dy + col0, r);
#pragma unroll
  for (int i = 0; i < NC / 4; ++i) sts128(dy_s + panel_off(row, col0 / 4 + i), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
}

// Sums c[0..N) over the warp and adds them to dst[0..N) (one coalesced reduction; dst belongs to this warp alone)
template <int N>
__device__ __forceinline__ void warp_reduce_red(const float* c, float* dst, int lane) {
  static_assert(N <= 32, "one lane per value");
  float mine = 0.f;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float v = c[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == i) mine = v;
  }
  if (lane < N) red_add(dst + lane, mine);
}

// dW accumulator of a step (TMEM lane = input feature m, column = output feature n) -> part[n * kw + m]
__device__ __forceinline__ void flush_dw(unsigned t_w, float* __restrict__ part, int N, int kw, int quarter, int half, int lane) {
  if (quarter * 32 >= kw) return;
  const int m = quarter * 32 + lane;
  for (int c = half; c * 16 < N; c += 2) {
    unsigned r[16];
    tmem_ld16(t_w + c * 16, r);
    tmem_wait_ld();
    float* dst = part + (c * 16) * kw + m;
#pragma unroll
    for (int j = 0; j < 16; ++j) red_add(dst + j * kw, __uint_as_float(r[j]));
  }
}

__global__ void __launch_bounds__(THREADS, 1)
reads_backward_tc_kernel(const __grid_constant__ PmtModelDesc D, const __grid_constant__ TcPlan TP, const __grid_constant__ TcBwdArgs A,
                         int n_stages, int stage_bytes) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // carve: [operand buffers 2 slots][weight ring][xch 2 slots][3 per-variant tables x 2 slots][pair exchange][block scalars][HeadConst][SharedB]
  unsigned char* p = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const unsigned opbuf = smem_addr(p); p += 2 * OPBUF_BYTES;
  const unsigned ring = smem_addr(p); p += (size_t)n_stages * stage_bytes;
  const unsigned xch_all = smem_addr(p); p += 2 * BXCH_ROWS * XCH_LD * sizeof(float);
  const unsigned tab_all = smem_addr(p); p += 2 * 3 * BW_TAB * sizeof(float);
  const unsigned pairx_all = smem_addr(p); p += 2 * 2 * TILE * 4 * sizeof(float);
  float* blkc = reinterpret_cast<float*>(p); p += PMT_MAX_BLOCKS * BC_STRIDE * sizeof(float);
  HeadConst* HC = reinterpret_cast<HeadConst*>(p); p += sizeof(HeadConst);
  SharedB* S = reinterpret_cast<SharedB*>((reinterpret_cast<uintptr_t>(p) + 15) & ~uintptr_t(15));

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int lane = tid & 31;
  const float* W = A.wflat;
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_addr(&S->bar_a[s]), 8); mbar_init(smem_addr(&S->bar_d[s]), 1); mbar_init(smem_addr(&S->bar_w[s]), 1);
      mbar_init(smem_addr(&S->act_full[s]), 1); mbar_init(smem_addr(&S->act_free[s]), 9);
    }
    for (int i = 0; i < n_stages; ++i) { mbar_init(smem_addr(&S->wfull[i]), 1); mbar_init(smem_addr(&S->wfree[i]), 2); }
    fence_mbar_init();
    head_constants(D, W, HC);
  }
  for (int i = tid; i < D.n_blocks * BC_STRIDE; i += THREADS) {
    const PmtBlockOffsets& BO = D.blocks[i / BC_STRIDE];
    const int c = i % BC_STRIDE, H = D.d_ffn / 2;
    float v = 0.f;
    if (c < BC_LN2B) { if (c < H) v = W[BO.ln2_w + c]; }
    else if (c < BC_REG) { if (c - BC_LN2B < H) v = W[BO.ln2_b + c - BC_LN2B]; }
    else if (c < BC_AREF) { if (c - BC_REG < H) v = W[BO.regularizer + c - BC_REG]; }
    else if (c == BC_AREF) v = W[BO.alpha_ref];
    else if (c == BC_AALT) v = W[BO.alpha_alt];
    else if (c == BC_BREF) v = W[BO.beta_ref];
    else if (c == BC_BALT) v = W[BO.beta_alt];
    else if (c == BC_GAMMA) v = W[BO.gamma];
    else if (c == BC_REGW) v = W[BO.reg_weight] + 0.25f;   // gated_mlp.py:237
    blkc[i] = v;
  }
  if (warp == MMA_WARP) tmem_alloc<TMEM_COLS>(smem_addr(&S->tmem_base));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const int tile_first = A.tile_first;
  const int n_tiles = min(__ldg(A.tiles), A.tile_limit) - tile_first;
  const int n_slots = 2 * gridDim.x;
  // tile t of the range goes to slot (t % n_slots): slot 0 of every CTA first, then slot 1; every slot of the CTA runs
  // the same number of rounds (an idle slot walks an empty tile over the scratch of tile 0)
  const int rounds = n_tiles > (int)blockIdx.x ? (n_tiles - (int)blockIdx.x + n_slots - 1) / n_slots : 0;
  const int n_steps = TP.n_steps;
  const unsigned tmem_base = __shfl_sync(0xffffffffu, S->tmem_base, 0);

  if (warp == LOAD_WARP) {
    if (lane == 0) {
      // ===================================== transposed weight images =====================================
      int stage = 0;
      unsigned parity = 1;   // first pass through the ring: stages are free
      for (int round = 0; round < rounds; ++round)
        for (int step = n_steps - 1; step >= 1; --step) {
          const TcStep& o = TP.step[step];
          mbar_wait(smem_addr(&S->wfree[stage]), parity);
          mbar_expect_tx(smem_addr(&S->wfull[stage]), o.t_img_bytes);
          bulk_g2s(ring + stage * stage_bytes, A.image_t + o.t_img_off, o.t_img_bytes, smem_addr(&S->wfull[stage]));
          if (++stage == n_stages) { stage = 0; parity ^= 1; }
        }
    } else if (lane <= 2) {
      // ===================================== saved operands of one slot =====================================
      const int s = lane - 1;
      unsigned parity = 1;
      for (int round = 0; round < rounds; ++round) {
        const int t = (int)blockIdx.x + s * (int)gridDim.x + round * n_slots;
        const unsigned char* src = A.scratch + (size_t)(t < n_tiles ? t : 0) * TP.tile_bytes;
        for (int step = n_steps - 1; step >= 0; --step) {
          const TcStep& o = TP.step[step];
          mbar_wait(smem_addr(&S->act_free[s]), parity);
          parity ^= 1;
          mbar_expect_tx(smem_addr(&S->act_full[s]), o.scr_bytes);
          bulk_g2s(opbuf + s * OPBUF_BYTES, src + o.scr_off, o.scr_bytes, smem_addr(&S->act_full[s]));
        }
      }
    }
    __syncwarp();
  } else if (warp >= MMA_WARP) {
    // ===================================== MMA issuers: one warp per slot =====================================
    const int s = warp - MMA_WARP;
    const unsigned tb = tmem_base + s * SLOT_COLS;
    const unsigned bar_a = smem_addr(&S->bar_a[s]), bar_d = smem_addr(&S->bar_d[s]), bar_w = smem_addr(&S->bar_w[s]);
    const unsigned act_full = smem_addr(&S->act_full[s]), act_free = smem_addr(&S->act_free[s]);
    const uint64_t a_desc = desc_panels(opbuf + s * OPBUF_BYTES, PANEL_BYTES);
    const uint64_t b_desc = desc_panels(opbuf + s * OPBUF_BYTES + 2 * PANEL_BYTES, PANEL_BYTES);
    int stage = 0;
    unsigned wparity = 0, aparity = 0, fparity = 0;
    for (int round = 0; round < rounds; ++round) {
      for (int step = n_steps - 1; step >= 0; --step) {
        const TcStep& o = TP.step[step];
        const int oN = o.N, oNd = o.Nd, oKSd = o.KSd;
        if (step > 0) mbar_wait(smem_addr(&S->wfull[stage]), wparity);
        mbar_wait(bar_a, aparity);
        aparity ^= 1;
        tc_fence_after();
        if (elect_one()) {
          if (step > 0) {   // data gradient: D[128 x Nd] = dY[128 x N] . W^T image
            const unsigned idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(oNd >> 3) << 17) | ((128u >> 4) << 24);
            const uint64_t b_hi = smem_desc(ring + stage * stage_bytes);
            const unsigned kb_stride16 = (unsigned)(oNd * 128) >> 4;
            switch (oKSd) {
              case 2: issue_chain<2, 1>(tb + COL_D, tb + COL_DY, 0u, b_hi, 0ull, kb_stride16, idesc, 0u, false); break;
              case 4: issue_chain<4, 1>(tb + COL_D, tb + COL_DY, 0u, b_hi, 0ull, kb_stride16, idesc, 0u, false); break;
              case 6: issue_chain<6, 1>(tb + COL_D, tb + COL_DY, 0u, b_hi, 0ull, kb_stride16, idesc, 0u, false); break;
              default: issue_chain<8, 1>(tb + COL_D, tb + COL_DY, 0u, b_hi, 0ull, kb_stride16, idesc, 0u, false); break;
            }
            mma_commit(smem_addr(&S->wfree[stage]));
          }
          mma_commit(bar_d);
        }
        __syncwarp();
        if (step > 0 && ++stage == n_stages) { stage = 0; wparity ^= 1; }
        mbar_wait(act_full, fparity);
        fparity ^= 1;
        tc_fence_after();
        if (elect_one()) {   // weight gradient: DW[m][n] = sum over the tile's rows of operand[r][m] * dY[r][n]
          const unsigned idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((unsigned)(oN >> 3) << 17) | ((128u >> 4) << 24);
#pragma unroll
          for (int ks = 0; ks < TILE / 8; ++ks)
            mma_ss_desc64(tb + COL_DW, a_desc + (uint64_t)(ks * 64), b_desc + (uint64_t)(ks * 64), idesc, ks > 0 ? 1u : 0u);
          mma_commit(bar_w);
          mma_commit(act_free);
        }
        __syncwarp();
      }
    }
  } else {
    // ============ epilogue: two threads per row; thread (row, half) owns half of the row's columns ============
    const int slot = warp >> 3, half = (warp >> 2) & 1, quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int srow = half * TILE + row;
    const int slot_bar = 1 + slot, pair_bar = 3 + slot * 4 + quarter;
    SlotMeta* M = &S->slot[slot];
    const unsigned m_rowvar = smem_addr(M->rowvar), m_ref_start = smem_addr(M->ref_start), m_ref_cnt = smem_addr(M->ref_cnt),
                   m_alt_start = smem_addr(M->alt_start), m_alt_cnt = smem_addr(M->alt_cnt);
    const unsigned xch = xch_all + slot * BXCH_ROWS * XCH_LD * 4;
    const unsigned t_means = tab_all + slot * 3 * BW_TAB * 4, t_dmr = t_means + BW_TAB * 4, t_creg = t_dmr + BW_TAB * 4;
    const unsigned px_mine = pairx_all + ((slot * 2 + half) * TILE + row) * 16, px_other = pairx_all + ((slot * 2 + (half ^ 1)) * TILE + row) * 16;
    const unsigned bar_a = smem_addr(&S->bar_a[slot]), bar_d = smem_addr(&S->bar_d[slot]), bar_w = smem_addr(&S->bar_w[slot]);
    const unsigned act_full = smem_addr(&S->act_full[slot]), act_free = smem_addr(&S->act_free[slot]);
    const unsigned trow = tmem_base + slot * SLOT_COLS + ((unsigned)(quarter * 32) << 16);
    const unsigned t_g = trow + COL_G, t_d = trow + COL_D, t_dy = trow + COL_DY, t_w = trow + COL_DW;
    const unsigned act_s = opbuf + slot * OPBUF_BYTES, dy_s = act_s + 2 * PANEL_BYTES;
    const int E = D.d_feat, K = D.n_clusters, Dm = D.d_model, H = D.d_ffn / 2, DR = D.d_read;
    const int DIS = D.d_info + D.d_seq;
    const int n_half = half ? DIS : DR;
    const unsigned inv_h = (65536u + (unsigned)H - 1u) / (unsigned)H;
    float* const part = A.partials + (size_t)(2 * blockIdx.x + slot) * TP.part_floats;
    float* const scal = part + TP.scal_off + (half * 4 + quarter) * SCAL_W;
    unsigned dparity = 0, wparity = 0, fparity = 0;

    for (int round = 0; round < rounds; ++round) {
      const int t = (int)blockIdx.x + slot * (int)gridDim.x + round * n_slots;
      // ---------------- tile meta (as the forward) ----------------
      int v0 = 0, nv = 0;
      if (t < n_tiles) { v0 = __ldg(A.tiles + 2 + 2 * (tile_first + t)); nv = __ldg(A.tiles + 3 + 2 * (tile_first + t)); }
      const unsigned char* const scr = A.scratch + (size_t)(t < n_tiles ? t : 0) * TP.tile_bytes;
      int ref_pad = 0;
      if (half == 0) M->rowvar[row] = 255;
      named_barrier(slot_bar, 256);
      if (nv > 0) {
        const long long r_base = __ldg(A.batch.ref_off + v0), a_base = __ldg(A.batch.alt_off + v0);
        const long long nr_tot = __ldg(A.batch.ref_off + v0 + nv) - r_base;
        ref_pad = (int)((nr_tot + 3) & ~3LL);
        if (half == 0 && row < nv) {
          const long long r0 = __ldg(A.batch.ref_off + v0 + row), r1 = __ldg(A.batch.ref_off + v0 + row + 1);
          const long long a0 = __ldg(A.batch.alt_off + v0 + row), a1 = __ldg(A.batch.alt_off + v0 + row + 1);
          const int rs = (int)(r0 - r_base), rc = (int)(r1 - r0), as = ref_pad + (int)(a0 - a_base), ac = (int)(a1 - a0);
          M->ref_start[row] = (unsigned char)rs; M->ref_cnt[row] = (unsigned char)rc;
          M->alt_start[row] = (unsigned char)as; M->alt_cnt[row] = (unsigned char)ac;
          for (int i = 0; i < rc; ++i) M->rowvar[rs + i] = (unsigned char)row;
          for (int i = 0; i < ac; ++i) M->rowvar[as + i] = (unsigned char)row;
        }
      }
      named_barrier(slot_bar, 256);
      const int rv = (int)lds_u8(m_rowvar + row);
      const int my_var = rv == 255 ? -1 : rv;
      const bool real = my_var >= 0;
      const int mv = real ? my_var : 0;
      const bool is_alt = row >= ref_pad;
      const int my_ref_cnt = (int)lds_u8(m_ref_cnt + mv), my_alt_cnt = (int)lds_u8(m_alt_cnt + mv);
      const int owner_row = my_ref_cnt > 0 ? (int)lds_u8(m_ref_start + mv) : (int)lds_u8(m_alt_start + mv);   // one row per variant
      const long long vg = (long long)v0 + mv;

      for (int step = n_steps - 1; step >= -1; --step) {
        // E(step): dL/d(output of `step`) from the data gradient of step + 1; step == -1 only drains the pipeline
        const int bepi = step >= 0 ? TP.step[step].bepi : -1;
        const bool first = step == n_steps - 1;
        float dy[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) dy[i] = 0.f;
        if (!first) {
          mbar_wait(bar_d, dparity); dparity ^= 1;
          mbar_wait(act_full, fparity); fparity ^= 1;
          tc_fence_after();
        }
        switch (bepi) {
          case BE_HEAD: {   // feature_clustering.py:82-135 and the set means (artifact_model.py:291-292) in reverse
            const bool live = is_alt && real;
            float f[MAXE];
            {
              const float* fi = reinterpret_cast<const float*>(scr + TP.f_off) + row;
#pragma unroll
              for (int e = 0; e < MAXE; ++e) f[e] = e < E ? __ldg(fi + e * TILE) : 0.f;
            }
            const int n_logit = K + 2;
            if (half == 0) {
              const float g0 = (live && A.d_logits_bk) ? __ldg(A.d_logits_bk + vg * n_logit) : 0.f;
              const float g1 = (live && A.d_logits_bk) ? __ldg(A.d_logits_bk + vg * n_logit + 1) : 0.f;
              const float* dm = is_alt ? A.d_alt_means : A.d_ref_means;
              const float inv_cnt = 1.f / ((float)(is_alt ? my_alt_cnt : my_ref_cnt) + 1e-4f);
              float cs[MAXE];
#pragma unroll
              for (int e = 0; e < MAXE; ++e) {
                cs[e] = 0.f;
                if (e < E) {
                  const float s = HC->sigma[e], fe = f[e], is2 = 1.f / (s * s);
                  dy[e] = -g0 * fe * is2 - 0.25f * g1 * fe * is2;
                  cs[e] = g0 * (-1.f / s + fe * fe * is2 / s) + g1 * (-1.f / s + 0.25f * fe * fe * is2 / s);
                  if (real && dm) dy[e] += __ldg(dm + vg * E + e) * inv_cnt;
                }
              }
              warp_reduce_red<MAXE>(cs, scal + PMT_MAX_BLOCKS * SCAL_BLOCK, lane);
              named_barrier(pair_bar, 64);
#pragma unroll
              for (int e = 0; e < MAXE; ++e) dy[e] = (e < E && real) ? rna_tf32(dy[e] + lds_f32(xch + (e * XCH_LD + row) * 4)) : 0.f;
            } else {
              float dfb[MAXE];
#pragma unroll
              for (int e = 0; e < MAXE; ++e) dfb[e] = 0.f;
              for (int k = 0; k < K; ++k) {
                const float gk = (live && A.d_logits_bk) ? __ldg(A.d_logits_bk + vg * n_logit + 2 + k) : 0.f;
                const float* u = W + D.unit_ke + k * E;
                const float tau = __ldg(W + D.tau_k + k), lam = __ldg(W + D.lambda_k + k), sg = __ldg(W + D.emg_sigma_k + k),
                            mu = __ldg(W + D.mu_k + k);
                float pr = 0.f;
#pragma unroll
                for (int e = 0; e < MAXE; ++e) if (e < E) pr = fmaf(f[e], __ldg(u + e), pr);
                float o2 = 0.f, odu = 0.f;
#pragma unroll
                for (int e = 0; e < MAXE; ++e) if (e < E) { const float o = f[e] - pr * __ldg(u + e); o2 = fmaf(o, o, o2); odu = fmaf(o, __ldg(u + e), odu); }
                const float zarg = (HC->shift[k] - pr) / HC->sqrt2_sigma[k];
                const float dlp = dlogerfc(zarg);
                const float dpar_dp = -dlp / HC->sqrt2_sigma[k] - lam;
                const float c_orth = -1.f / HC->two_tau2[k];
                float c[HEAD_K_STRIDE];
#pragma unroll
                for (int e = 0; e < MAXE; ++e) {
                  c[e] = 0.f;
                  if (e < E) {
                    const float fe = f[e], ue = __ldg(u + e), o = fe - pr * ue;
                    dfb[e] += gk * (c_orth * (2.f * o - 2.f * odu * ue) + dpar_dp * ue);
                    c[e] = gk * (c_orth * (-2.f * fe * odu - 2.f * pr * o) + dpar_dp * fe);
                  }
                }
                c[MAXE + 0] = gk * (-(float)(E - 1) / tau + o2 / (tau * tau * tau));
                c[MAXE + 1] = gk * (dlp / HC->sqrt2_sigma[k] + lam);
                c[MAXE + 2] = gk * (dlp * (1.41421356237f * lam - zarg / sg) + lam * lam * sg);
                c[MAXE + 3] = gk * (1.f / lam + dlp * sg * 0.70710678118f + mu + lam * sg * sg - pr);
                // the log cluster weight is added once per variant, after the sum over its reads (feature_clustering.py:115-116)
                c[MAXE + 4] = (live && row == (int)lds_u8(m_alt_start + mv)) ? gk : 0.f;
                warp_reduce_red<HEAD_K_STRIDE>(c, scal + PMT_MAX_BLOCKS * SCAL_BLOCK + 16 + k * HEAD_K_STRIDE, lane);
              }
#pragma unroll
              for (int e = 0; e < MAXE; ++e) if (e < E) sts_f32(xch + (e * XCH_LD + row) * 4, dfb[e]);
              named_barrier(pair_bar, 64);
            }
          } break;
          case BE_GINIT64: {   // the last layer read the residual stream itself
            float v[32];
            load_cols<32>(t_d + half * 32, v);
            unsigned r[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) { v[i] = (real && i < n_half) ? v[i] : 0.f; r[i] = __float_as_uint(v[i]); dy[i] = rna_tf32(v[i]); }
            tmem_st32(t_g + half * 32, r);
          } break;
          case BE_DZ64:
          case BE_GACC64: {   // mlp.py:8-22 in reverse: through u = SELU / scale of the layer's input
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              float v[16], a[16];
              load_cols<16>(t_d + half * 32 + c * 16, v);
              load_act<16>(act_s, row, half * 32 + c * 16, a);
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] = (real && c * 16 + i < n_half) ? v[i] * du(a[i]) : 0.f;
              if (bepi == BE_GACC64) {
                float g[16];
                load_cols<16>(t_g + half * 32 + c * 16, g);
                unsigned r[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) { v[i] += g[i]; r[i] = __float_as_uint(v[i]); }
                tmem_st16(t_g + half * 32 + c * 16, r);
              }
#pragma unroll
              for (int i = 0; i < 16; ++i) dy[c * 16 + i] = rna_tf32(v[i]);
            }
          } break;
          case BE_DZ32:
          case BE_GACC32:
          case BE_FIRST: {
            float v[16], a[16];
            load_cols<16>(t_d + half * 16, v);
            load_act<16>(act_s, row, half * 16, a);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = (real && half * 16 + i < DR) ? v[i] * du(a[i]) : 0.f;
            if (bepi != BE_DZ32) {
              float g[16];
              load_cols<16>(t_g + half * 16, g);
              unsigned r[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) { v[i] += g[i]; r[i] = __float_as_uint(v[i]); }
              tmem_st16(t_g + half * 16, r);
            }
            if (bepi == BE_FIRST) {   // x0 = SELU(z0): the embedding's first layer (mlp.py:61-62)
              const float* x0 = reinterpret_cast<const float*>(scr + TP.x0_off) + (half * 16) * TILE + row;
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float x = __ldg(x0 + i * TILE);
                v[i] *= x > 0.f ? SELU_SCALE : x + SELU_SCALE * SELU_ALPHA;
              }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) dy[i] = rna_tf32(v[i]);
          } break;
          case BE_LN64:
          case BE_LN_EMBED: {   // LayerNorm of gated block `blk` in reverse (gated_mlp.py:185), added to the residual gradient
            const int blk = TP.step[step + 1].blk;
            const float rstd = __ldg(reinterpret_cast<const float*>(scr + TP.rstd_off) + blk * TILE + row);
            float p1 = 0.f, p2 = 0.f;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              float v[16], a[16];
              load_cols<16>(t_d + half * 32 + c * 16, v);
              load_act<16>(act_s, row, half * 32 + c * 16, a);
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (c * 16 + i < n_half) { p1 += v[i]; p2 = fmaf(v[i], a[i], p2); }
            }
            sts_f32x2(px_mine, p1, p2);
            named_barrier(pair_bar, 64);
            const float2 oth = lds_f32x2(px_other);
            const float m1 = (p1 + oth.x) / (float)Dm, m2 = (p2 + oth.y) / (float)Dm;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              float v[16], a[16], g[16];
              load_cols<16>(t_d + half * 32 + c * 16, v);
              load_act<16>(act_s, row, half * 32 + c * 16, a);
              load_cols<16>(t_g + half * 32 + c * 16, g);
              unsigned r[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                g[i] = (real && c * 16 + i < n_half) ? g[i] + rstd * (v[i] - m1 - a[i] * m2) : 0.f;
                r[i] = __float_as_uint(g[i]);
                dy[c * 16 + i] = g[i];
              }
              tmem_st16(t_g + half * 32 + c * 16, r);
            }
            if (bepi == BE_LN_EMBED) {
              // concat (artifact_model.py:246-251): columns 32.. of the stream are the variant's info/sequence embedding
              for (int pass = 0; pass < 2; ++pass) {
                if (half == 1) {
#pragma unroll
                  for (int i = 0; i < 16; ++i) sts_f32(xch + (i * XCH_LD + row) * 4, pass ? dy[16 + i] : dy[i]);
                }
                named_barrier(slot_bar, 256);
                for (int idx = srow; idx < nv * 16; idx += 256) {
                  const int j = idx >> 4, c = idx & 15, col = pass * 16 + c;
                  if (col < DIS) {
                    const int rs = (int)lds_u8(m_ref_start + j), rc = (int)lds_u8(m_ref_cnt + j), as = (int)lds_u8(m_alt_start + j),
                              ac = (int)lds_u8(m_alt_cnt + j);
                    float acc = 0.f;
                    for (int i = 0; i < rc; ++i) acc += lds_f32(xch + (c * XCH_LD + rs + i) * 4);
                    for (int i = 0; i < ac; ++i) acc += lds_f32(xch + (c * XCH_LD + as + i) * 4);
                    A.d_info_seq[((long long)v0 + j) * DIS + col] = acc;
                  }
                }
                named_barrier(slot_bar, 256);
              }
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) dy[i] = rna_tf32(dy[i]);
          } break;
          case BE_GATE: {   // spatial gating unit in reverse (gated_mlp.py:186-190, 228-251); this thread owns hidden units [k0, k0 + 6)
            const int blk = TP.step[step].blk;
            const unsigned bcs = smem_addr(blkc + blk * BC_STRIDE);
            const int k0 = half * 6;
            float dt[6];
            {
              unsigned r[24];
              tmem_ld16(t_d, r); tmem_ld8(t_d + 16, r + 16);
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 6; ++j) {
                const unsigned sel = half == 0 ? (is_alt ? r[6 + j] : r[j]) : (j < 5 ? (is_alt ? r[17 + j] : r[12 + j]) : 0u);
                dt[j] = __uint_as_float(sel);
              }
            }
            const float* gi = reinterpret_cast<const float*>(scr + TP.gate_off) + ((blk * GATE_ITEMS) * 2 + half) * TILE + row;
            float z1[6], xh2[6], ds2[6], dgate[6];
#pragma unroll
            for (int j = 0; j < 6; ++j) {
              const bool ok = real && k0 + j < H;
              z1[j] = ok ? __ldg(gi + j * 2 * TILE) : 0.f;
              xh2[j] = ok ? __ldg(gi + (6 + j) * 2 * TILE) : 0.f;
              ds2[j] = ok ? __ldg(gi + (12 + j) * 2 * TILE) : 0.f;
              dt[j] = ok ? dt[j] : 0.f;
              dgate[j] = dt[j] * z1[j];
              if (k0 + j < H) sts_f32(xch + ((k0 + j) * XCH_LD + row) * 4, dgate[j]);
            }
            const float rstd2 = real ? __ldg(gi + 18 * 2 * TILE) : 0.f;
            {
              const float* mg = reinterpret_cast<const float*>(scr + TP.means_off) + blk * BW_TAB;
              for (int i = srow; i < nv * 2 * MAXH; i += 256) sts_f32(t_means + i * 4, __ldg(mg + i));
            }
            named_barrier(slot_bar, 256);
            {   // mean fields in reverse (ragged_sets.py:144-155): one (variant, hidden unit) per thread
              const float regw = lds_f32(bcs + BC_REGW * 4), b_ref = lds_f32(bcs + BC_BREF * 4), b_alt = lds_f32(bcs + BC_BALT * 4),
                          gamma = lds_f32(bcs + BC_GAMMA * 4);
              for (int idx = srow; idx < nv * H; idx += 256) {
                const int j = (int)(((unsigned)idx * inv_h) >> 16), f = idx - j * H;
                const int rs = (int)lds_u8(m_ref_start + j), rc = (int)lds_u8(m_ref_cnt + j), as = (int)lds_u8(m_alt_start + j),
                          ac = (int)lds_u8(m_alt_cnt + j);
                float s_ref = 0.f, s_alt = 0.f;
                for (int i = 0; i < rc; ++i) s_ref += lds_f32(xch + (f * XCH_LD + rs + i) * 4);
                for (int i = 0; i < ac; ++i) s_alt += lds_f32(xch + (f * XCH_LD + as + i) * 4);
                const float dm_ref = b_ref * s_ref + gamma * s_alt, dm_alt = b_alt * s_alt;
                const float den_ref = (float)rc + regw, den_alt = (float)ac + 1e-4f;
                sts_f32(t_dmr + ((2 * j) * MAXH + f) * 4, dm_ref / den_ref);
                sts_f32(t_dmr + ((2 * j + 1) * MAXH + f) * 4, dm_alt / den_alt);
                sts_f32(t_creg + ((2 * j) * MAXH + f) * 4, dm_ref * regw / den_ref);
                sts_f32(t_creg + ((2 * j + 1) * MAXH + f) * 4,
                        dm_ref * (lds_f32(bcs + (BC_REG + f) * 4) - lds_f32(t_means + ((2 * j) * MAXH + f) * 4)) / den_ref);
              }
            }
            named_barrier(slot_bar, 256);
            const float alpha = lds_f32(bcs + (is_alt ? BC_AALT : BC_AREF) * 4);
            const float beta = lds_f32(bcs + (is_alt ? BC_BALT : BC_BREF) * 4);
            const float gamma = is_alt ? lds_f32(bcs + BC_GAMMA * 4) : 0.f;
            const int side = is_alt ? 1 : 0;
            const bool owner = real && row == owner_row;
            float c[SCAL_BLOCK];
            float s_alpha = 0.f, s_beta = 0.f, s_gamma = 0.f, c_regw = 0.f, q1 = 0.f, q2 = 0.f;
            float dz1[6], dxh2[6];
#pragma unroll
            for (int j = 0; j < 6; ++j) {
              const bool ok = real && k0 + j < H;
              const int f = ok ? k0 + j : 0;
              const float ln2w = lds_f32(bcs + (BC_LN2W + f) * 4), ln2b = lds_f32(bcs + (BC_LN2B + f) * 4);
              const float z2n = fmaf(xh2[j], ln2w, ln2b);
              const float m_ref = ok ? lds_f32(t_means + ((2 * mv) * MAXH + f) * 4) : 0.f;
              const float m_own = ok ? lds_f32(t_means + ((2 * mv + side) * MAXH + f) * 4) : 0.f;
              const float gate = fmaf(beta, m_own, fmaf(gamma, m_ref, fmaf(z2n, alpha, 1.f)));
              dz1[j] = ok ? dt[j] * gate * (z1[j] > 0.f ? SELU_SCALE : z1[j] + SELU_SCALE * SELU_ALPHA) : 0.f;
              s_alpha = fmaf(dgate[j], z2n, s_alpha);
              s_beta = fmaf(dgate[j], m_own, s_beta);
              s_gamma = fmaf(dgate[j], m_ref, s_gamma);
              const float dz2n = ok ? fmaf(alpha, dgate[j], lds_f32(t_dmr + ((2 * mv + side) * MAXH + f) * 4)) : 0.f;
              c[6 + j] = dz2n * xh2[j];
              c[12 + j] = dz2n;
              c[18 + j] = (owner && ok) ? lds_f32(t_creg + ((2 * mv) * MAXH + f) * 4) : 0.f;
              c_regw += (owner && ok) ? lds_f32(t_creg + ((2 * mv + 1) * MAXH + f) * 4) : 0.f;
              dxh2[j] = dz2n * ln2w;
              q1 += dxh2[j];
              q2 = fmaf(dxh2[j], xh2[j], q2);
            }
            c[0] = is_alt ? 0.f : s_alpha; c[1] = is_alt ? s_alpha : 0.f;
            c[2] = is_alt ? 0.f : s_beta;  c[3] = is_alt ? s_beta : 0.f;
            c[4] = is_alt ? s_gamma : 0.f; c[5] = c_regw;
            warp_reduce_red<SCAL_BLOCK>(c, scal + blk * SCAL_BLOCK, lane);
            // SGU LayerNorm in reverse: its statistics run over all H hidden units of the row (both threads)
            sts_f32x2(px_mine + 8, q1, q2);
            named_barrier(pair_bar, 64);
            const float2 oth = lds_f32x2(px_other + 8);
            const float m1 = (q1 + oth.x) / (float)H, m2 = (q2 + oth.y) / (float)H;
            // dY columns of this thread: [ref z1 (6) | ref z2 (6) | alt z1 (6) | alt z2 (6)]
#pragma unroll
            for (int j = 0; j < 6; ++j) {
              const bool ok = real && k0 + j < H;
              const float dz2 = ok ? rstd2 * (dxh2[j] - m1 - xh2[j] * m2) * ds2[j] : 0.f;
              const float a = rna_tf32(dz1[j]), b = rna_tf32(dz2);
              dy[j] = is_alt ? 0.f : a; dy[6 + j] = is_alt ? 0.f : b;
              dy[12 + j] = is_alt ? a : 0.f; dy[18 + j] = is_alt ? b : 0.f;
            }
          } break;
          default: break;
        }
        if (!first) {
          // the operand of step + 1 has been read; its weight gradient must have left shared memory and TMEM before
          // this step's dY and dW overwrite them
          __syncwarp();
          if (lane == 0) mbar_arrive(act_free);
          mbar_wait(bar_w, wparity); wparity ^= 1;
          tc_fence_after();
          const TcStep& prev = TP.step[step + 1];
          flush_dw(t_w, part + prev.part_off, prev.N, prev.kw, quarter, half, lane);
        }
        if (step < 0) break;
        switch (bepi) {
          case BE_HEAD: if (half == 0) store_dy<16>(t_dy, dy_s, row, 0, dy); break;
          case BE_LN_EMBED: if (half == 0) store_dy<32>(t_dy, dy_s, row, 0, dy); break;
          case BE_GATE: store_dy<24>(t_dy, dy_s, row, half * 24, dy); break;
          case BE_DZ32:
          case BE_GACC32:
          case BE_FIRST: store_dy<16>(t_dy, dy_s, row, half * 16, dy); break;
          default: store_dy<32>(t_dy, dy_s, row, half * 32, dy); break;
        }
        tmem_wait_st();
        fence_proxy_async();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_a);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc<TMEM_COLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// Transposed weight images for the data gradient: B[n' = operand column][k' = output column] = W'[k'][n'] of the
// folded forward weights, K-major with the 128-byte swizzle like the forward images, TF32 rounded to nearest.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int bwd_out_col(const PmtModelDesc& D, const TcStep& o, int nb) {   // backward dY column -> forward output column
  return o.pk == PK_PROJ1 ? proj1_bwd_col(nb, D.d_ffn / 2) : nb;
}

__global__ void pack_tc_bwd_kernel(const __grid_constant__ PmtModelDesc D, const __grid_constant__ TcPlan TP, const float* __restrict__ w,
                                   unsigned char* __restrict__ image) {
  const TcStep& o = TP.step[blockIdx.x];
  if (o.t_img_bytes == 0) return;
  const int Kp = o.N;                      // reduction length: output columns of the forward layer
  const int n_kb = (Kp + 31) / 32;
  for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < n_kb * o.Nd * 32; idx += gridDim.y * blockDim.x) {
    const int kb = idx / (o.Nd * 32), rem = idx % (o.Nd * 32), n = rem / 32, kk = rem % 32;
    const int k = kb * 32 + kk;
    float v = 0.f;
    if (k < Kp && n < o.KS * 8) {
      const int nf = bwd_out_col(D, o, k);
      if (nf >= 0) v = tc_weight(D, o, w, nf, n);
    }
    const unsigned L = (unsigned)n * 128u + (unsigned)kk * 4u;
    const unsigned phys = L ^ (((L >> 7) & 7u) << 4);
    *reinterpret_cast<float*>(image + (size_t)o.t_img_off + (size_t)kb * o.Nd * 128 + phys) = rna_tf32(v);
  }
}

// ------------------------------------------------------------------------------------------------
// Private gradient buffers -> flat gradient.  reduce: fixed-order sum over the (CTA, slot) buffers.  unfold: the image
// gradients dI[step][n][k] through the folds of tc_weight(), every flat parameter written by exactly one thread.
// ------------------------------------------------------------------------------------------------
__global__ void reduce_private_kernel(const float* __restrict__ partials, int n_buf, int part_floats, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= part_floats) return;
  float s = 0.f;
  for (int b = 0; b < n_buf; ++b) s += partials[(size_t)b * part_floats + i];
  out[i] = s;
}

__device__ __forceinline__ float dimg(const float* __restrict__ g, const TcStep& o, int n, int k) { return g[o.part_off + n * o.kw + k]; }

// blocks [0, n_steps): one per step; blocks [n_steps, n_steps + n_blocks): the scalars of a gated block; last block: head
__global__ void unfold_kernel(const __grid_constant__ PmtModelDesc D, const __grid_constant__ TcPlan TP, const float* __restrict__ w,
                              const float* __restrict__ g, float* __restrict__ out) {
  const int DR = D.d_read, Dm = D.d_model, H = D.d_ffn / 2, E = D.d_feat, K = D.n_clusters;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int b = blockIdx.x;
  if (b < TP.n_steps) {
    const TcStep& o = TP.step[b];
    switch (o.pk) {
      case PK_LINEAR: {
        // image = alpha * (scale) * W; for the last layer of a DenseSkipBlock the un-scaled U goes out (skip_fix_kernel
        // turns it into dW = alpha U and d alpha = <W, U> + <b, Ub>), which is scale * dI either way
        const float sc = o.k_selu_scale ? SELU_SCALE : 1.f;
        for (int i = tid; i < o.n_real * o.k_real; i += nt) {
          const int nn = i / o.k_real, kk = i % o.k_real;
          const int n = o.n_perm ? perm64(nn, DR) : nn, k = o.k_perm ? perm64(kk, DR) : kk;
          out[o.w_off + i] += sc * dimg(g, o, n, k);
        }
        for (int nn = tid; nn < o.n_real; nn += nt) out[o.b_off + nn] += dimg(g, o, o.n_perm ? perm64(nn, DR) : nn, o.bias_col);
      } break;
      case PK_PROJ1: {   // image[n][k] = W1[nn][kk] ln_w[kk]; bias column: b1[nn] + sum_j W1[nn][j] ln_b[j]
        const PmtBlockOffsets& BO = D.blocks[o.blk];
        for (int i = tid; i < 2 * 2 * H * Dm; i += nt) {
          const int set = i / (2 * H * Dm), r = i % (2 * H * Dm), nn = r / Dm, kk = r % Dm;
          const int unit = nn % H, z2 = nn / H, h = unit / 6;
          const int nb = 24 * h + 12 * set + 6 * z2 + unit % 6;
          const int k = perm64(kk, DR);
          out[(set ? BO.p1_alt_w : BO.p1_ref_w) + nn * Dm + kk] += dimg(g, o, nb, k) * w[BO.ln_w + kk] + dimg(g, o, nb, o.bias_col) * w[BO.ln_b + kk];
        }
        for (int i = tid; i < 2 * 2 * H; i += nt) {
          const int set = i / (2 * H), nn = i % (2 * H), unit = nn % H, z2 = nn / H;
          const int nb = 24 * (unit / 6) + 12 * set + 6 * z2 + unit % 6;
          out[(set ? BO.p1_alt_b : BO.p1_ref_b) + nn] += dimg(g, o, nb, o.bias_col);
        }
        for (int kk = tid; kk < Dm; kk += nt) {
          const int k = perm64(kk, DR);
          float dw = 0.f, db = 0.f;
          for (int set = 0; set < 2; ++set)
            for (int nn = 0; nn < 2 * H; ++nn) {
              const int unit = nn % H, z2 = nn / H;
              const int nb = 24 * (unit / 6) + 12 * set + 6 * z2 + unit % 6;
              const float wv = w[(set ? BO.p1_alt_w : BO.p1_ref_w) + nn * Dm + kk];
              dw = fmaf(dimg(g, o, nb, k), wv, dw);
              db = fmaf(dimg(g, o, nb, o.bias_col), wv, db);
            }
          out[BO.ln_w + kk] += dw;
          out[BO.ln_b + kk] += db;
        }
      } break;
      case PK_PROJ2: {   // operand: [t_ref k 0..5 | t_alt k 0..5 | t_ref k 6..10 | t_alt k 6..10 | is_ref | is_alt]
        const PmtBlockOffsets& BO = D.blocks[o.blk];
        for (int i = tid; i < 2 * Dm * H; i += nt) {
          const int set = i / (Dm * H), r = i % (Dm * H), nn = r / H, unit = r % H;
          const int k = unit < 6 ? (set ? 6 : 0) + unit : 12 + (set ? 5 : 0) + (unit - 6);
          out[(set ? BO.p2_alt_w : BO.p2_ref_w) + nn * H + unit] += dimg(g, o, perm64(nn, DR), k);
        }
        for (int i = tid; i < 2 * Dm; i += nt) {
          const int set = i / Dm, nn = i % Dm;
          out[(set ? BO.p2_alt_b : BO.p2_ref_b) + nn] += dimg(g, o, perm64(nn, DR), 22 + set);
        }
      } break;
      case PK_FINAL: {   // image[n][k] = sum_j Q[n][j] Wl[j][kk]; bias column: sum_j Q[n][j] (b[j] + t[j])
        for (int i = tid; i < E * o.k_real; i += nt) {
          const int j = i / o.k_real, kk = i % o.k_real, k = perm64(kk, DR);
          float s = 0.f;
          for (int n = 0; n < E; ++n) s = fmaf(w[D.rotation + n * E + j], dimg(g, o, n, k), s);
          out[o.w_off + i] += s;
        }
        for (int j = tid; j < E; j += nt) {
          float s = 0.f;
          for (int n = 0; n < E; ++n) s = fmaf(w[D.rotation + n * E + j], dimg(g, o, n, o.bias_col), s);
          out[o.b_off + j] += s;
          out[D.translation + j] += s;
        }
        for (int i = tid; i < E * E; i += nt) {
          const int n = i / E, j = i % E;
          float s = dimg(g, o, n, o.bias_col) * (w[o.b_off + j] + w[D.translation + j]);
          for (int kk = 0; kk < o.k_real; ++kk) s = fmaf(dimg(g, o, n, perm64(kk, DR)), w[o.w_off + j * o.k_real + kk], s);
          out[D.rotation + i] += s;
        }
      } break;
    }
    return;
  }
  // per-warp scalar slots: warp = half * 4 + quarter
  const float* sc = g + TP.scal_off;
  if (b < TP.n_steps + D.n_blocks) {
    const int blk = b - TP.n_steps;
    const PmtBlockOffsets& BO = D.blocks[blk];
    if (tid < 6) {
      float s = 0.f;
      for (int wp = 0; wp < 8; ++wp) s += sc[wp * SCAL_W + blk * SCAL_BLOCK + tid];
      const int off = tid == 0 ? BO.alpha_ref : (tid == 1 ? BO.alpha_alt : (tid == 2 ? BO.beta_ref : (tid == 3 ? BO.beta_alt : (tid == 4 ? BO.gamma : BO.reg_weight))));
      out[off] += s;
    }
    for (int i = tid; i < 3 * H; i += nt) {
      const int which = i / H, f = i % H, h = f / 6;
      float s = 0.f;
      for (int q = 0; q < 4; ++q) s += sc[(h * 4 + q) * SCAL_W + blk * SCAL_BLOCK + 6 + which * 6 + f % 6];
      out[(which == 0 ? BO.ln2_w : (which == 1 ? BO.ln2_b : BO.regularizer)) + f] += s;
    }
    return;
  }
  const int hb = PMT_MAX_BLOCKS * SCAL_BLOCK;
  for (int e = tid; e < E; e += nt) {
    float s = 0.f;
    for (int q = 0; q < 4; ++q) s += sc[q * SCAL_W + hb + e];
    out[D.sigma_e + e] += s;
  }
  for (int i = tid; i < K * (E + 5); i += nt) {
    const int k = i / (E + 5), r = i % (E + 5);
    float s = 0.f;
    for (int q = 0; q < 4; ++q) s += sc[(4 + q) * SCAL_W + hb + 16 + k * HEAD_K_STRIDE + (r < E ? r : MAXE + (r - E))];
    int off;
    if (r < E) off = D.unit_ke + k * E + r;
    else if (r == E) off = D.tau_k + k;
    else if (r == E + 1) off = D.mu_k + k;
    else if (r == E + 2) off = D.emg_sigma_k + k;
    else if (r == E + 3) off = D.lambda_k + k;
    else off = D.logw_k + k;
    out[off] += s;
  }
}

}  // namespace tc
}  // namespace pmt

// ================================================================================================
// host side
// ================================================================================================
using namespace pmt;
using namespace pmt::tc;

long long pmt_train_tile_bound(const PmtBatch* batch, int n_claims) {
  // without a row count (n_rows <= 0) nothing bounds the rows per variant: a training tile holds at least one whole set
  if (batch->n_rows <= 0) return batch->n_variants < 1 ? 1 : batch->n_variants;
  const long long rows = batch->n_rows;
  // a tile is closed when the next set does not fit or it holds BWD_MAXV sets; the last tile of a claim may be short
  long long bound = 2 * rows / TILE + batch->n_variants / BWD_MAXV + n_claims + 8;
  if (batch->max_rows_per_variant > 0) {
    // with the longest set known: a tile closed because the next set did not fit holds more than TILE - 3 - longest rows
    const long long longest = batch->max_rows_per_variant < TILE - 4 ? batch->max_rows_per_variant : TILE - 4;
    const long long tight = rows / (TILE - 3 - longest) + batch->n_variants / BWD_MAXV + n_claims + 8;
    if (tight < bound) bound = tight;
  }
  if (bound > batch->n_variants) bound = batch->n_variants;
  return bound < 1 ? 1 : bound;
}

// The operand scratch is sized from an upper bound of the tile count (pmt_train_tile_bound): should the planner ever produce more
// tiles than that, fail loudly instead of writing past the buffer.
__global__ void check_tile_bound_kernel(const int* __restrict__ tiles, int bound) {
  if (tiles[0] > bound) {
    printf("permutect_b200: %d tiles planned, bound %d (pmt_tc_bwd.cu: tile_bound)\n", tiles[0], bound);
    __trap();
  }
}

// The backward kernel's weight ring: as many stages as fit next to the fixed carve, at most NS_MAX.
Ring pmt_tc_bwd_ring(const TcPlan& T) {
  const size_t fixed = 2 * OPBUF_BYTES + 2 * BXCH_ROWS * XCH_LD * sizeof(float) + 2 * 3 * BW_TAB * sizeof(float) + 2 * 2 * TILE * 4 * sizeof(float) +
                       PMT_MAX_BLOCKS * BC_STRIDE * sizeof(float) + sizeof(HeadConst) + sizeof(SharedB) + 1024 + 64;
  Ring R;
  R.stage_bytes = (T.t_stage_bytes + 1023) & ~1023;
  R.n_stages = (int)((227 * 1024 - fixed) / R.stage_bytes);
  if (R.n_stages > NS_MAX) R.n_stages = NS_MAX;
  R.smem = fixed + (size_t)R.n_stages * R.stage_bytes;
  return R;
}

// The training forward of the tile-sized sets: deterministic tile list, then the SAVE variant of the read kernel over ALL
// tiles with the outputs switched on: the weight images are packed into W.tc_image, the tile list and the operands go to
// the saved buffer.
int pmt_tc_forward_train(const CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out, const FwdBuffers& W,
                         const SavedBuffers& S, cudaStream_t st) {
  const TcPlan& T = C.T;
  const long long bound = C.saved.bound;
  int n_claims = 0;
  if (pmt_plan_tiles(batch, BWD_MAXV, true, PMT_PARTIAL_CTAS, S.tiles, W.claims, &n_claims, st)) return 1;
  check_tile_bound_kernel<<<1, 1, 0, st>>>(S.tiles, (int)bound);
  if (pmt_launch_pack_tc(C.P, T, weights, W.tc_image, st)) return 1;
  const int grid = pmt_tile_grid(batch, n_claims, C.n_sm < PMT_PARTIAL_CTAS ? C.n_sm : PMT_PARTIAL_CTAS);
  TcArgs F;
  memset(&F, 0, sizeof(F));
  F.wflat = weights; F.image = W.tc_image; F.tiles = S.tiles; F.perm = nullptr; F.batch = *batch; F.out = *out;
  F.scratch = S.scratch; F.tile_first = 0; F.tile_limit = (int)bound;
  pmt_profile_begin(st);
  const int rc = pmt_launch_reads_tc_save(C, F, grid, st);
  pmt_profile_end(st);
  return rc;
}

// Backward of the tile-sized read sets: writes d_info_seq for the variants of those sets and leaves the weight gradients
// in the private buffers of the workspace; pmt_finish_reads_tc_backward adds them to d_weights.
int pmt_launch_reads_tc_backward(const CallPlan& C, const float* weights, const PmtBatch* batch, const float* info_seq,
                                 const float* d_logits_bk, const float* d_alt_means, const float* d_ref_means, float* d_info_seq,
                                 const TcBwdBuffers& W, int* grid_out, cudaStream_t st, const SavedBuffers* saved) {
  const TcPlan& T = C.T;
  const BwdLayout& L = C.tc_bwd;
  int* tiles = W.tiles;
  unsigned char* scratch = W.scratch;
  int n_claims = 0;
  if (saved) {   // the training forward left the tile list and every tile's operands (pmt_tc_forward_train): no recompute
    tiles = saved->tiles;
    scratch = saved->scratch;
    n_claims = L.n_claims;
  } else {
    if (pmt_plan_tiles(batch, BWD_MAXV, true, PMT_PARTIAL_CTAS, tiles, W.claims, &n_claims, st)) return 1;
    if (pmt_launch_pack_tc(C.P, T, weights, W.image_f, st)) return 1;
  }
  pack_tc_bwd_kernel<<<dim3(T.n_steps, 8), 256, 0, st>>>(C.P.d, T, weights, W.image_t);

  const int grid = pmt_tile_grid(batch, n_claims, C.n_sm < PMT_PARTIAL_CTAS ? C.n_sm : PMT_PARTIAL_CTAS);
  PMT_CUDA(cudaMemsetAsync(W.partials, 0, (size_t)2 * grid * T.part_floats * sizeof(float), st));
  const Ring& R = C.ring_bwd;
  PMT_CUDA(cudaFuncSetAttribute(reads_backward_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R.smem));

  PmtOutputs no_out;
  memset(&no_out, 0, sizeof(no_out));
  no_out.info_seq_be = const_cast<float*>(info_seq);   // read by the first gated block's concat
  TcArgs F;
  F.wflat = weights; F.image = W.image_f; F.tiles = tiles; F.perm = nullptr; F.batch = *batch; F.out = no_out; F.scratch = scratch;
  TcBwdArgs Bk;
  Bk.wflat = weights; Bk.image_t = W.image_t; Bk.tiles = tiles; Bk.batch = *batch; Bk.d_logits_bk = d_logits_bk;
  Bk.d_alt_means = d_alt_means; Bk.d_ref_means = d_ref_means; Bk.d_info_seq = d_info_seq; Bk.scratch = scratch; Bk.partials = W.partials;
  pmt_profile_begin(st);
  for (int c = 0; c < L.n_chunks; ++c) {
    F.tile_first = Bk.tile_first = c * L.chunk_tiles;
    F.tile_limit = Bk.tile_limit = (c + 1) * L.chunk_tiles;
    if (saved) Bk.scratch = scratch + (size_t)Bk.tile_first * T.tile_bytes;   // the kernel indexes a pass's scratch from its first tile
    else if (pmt_launch_reads_tc_save(C, F, grid, st)) return 1;
    reads_backward_tc_kernel<<<grid, THREADS, R.smem, st>>>(C.P.d, T, Bk, R.n_stages, R.stage_bytes);
  }
  pmt_profile_end(st);
  *grid_out = grid;
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "tensor-core backward launch failed: %s", cudaGetErrorString(e));
  return 0;
}

// d_weights += the tile-sized sets' gradient (call after the other kernels' sums have been WRITTEN to d_weights and before
// skip_fix_kernel: the last layer of a DenseSkipBlock is handed over un-scaled, as the SIMT kernels do).
int pmt_finish_reads_tc_backward(const CallPlan& C, const float* weights, float* d_weights, const TcBwdBuffers& W, int grid,
                                 cudaStream_t st) {
  const TcPlan& T = C.T;
  reduce_private_kernel<<<(T.part_floats + 255) / 256, 256, 0, st>>>(W.partials, 2 * grid, T.part_floats, W.reduced);
  unfold_kernel<<<T.n_steps + C.P.d.n_blocks + 1, 256, 0, st>>>(C.P.d, T, weights, W.reduced, d_weights);
  cudaError_t e = cudaGetLastError();
  PMT_CHECK(e == cudaSuccess, "tensor-core backward (unfold) launch failed: %s", cudaGetErrorString(e));
  return 0;
}
