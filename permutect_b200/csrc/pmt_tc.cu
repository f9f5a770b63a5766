// Tensor-core (tcgen05 / TMEM) forward of the read path for sm_100a.
//
// One persistent CTA per SM keeps TWO tiles of 128 reads in flight (ping-pong): while the tensor core runs a
// layer of tile A, the epilogue warps of tile B turn the previous accumulator into the next operand.
//
//   warps 0-7   epilogue of slot 0: two threads per read (row) r of the tile -- TMEM lane r, 32 columns each
//   warps 8-15  epilogue of slot 1
//   warps 16-17 MMA issuers, one per slot: warp-uniform loop, one elected lane issues the tcgen05.mma chains
//               (kind::tf32, M = 128, A operand in TMEM, B = weights in shared memory) and commits to mbarriers
//   warp  18    weight loader: streams every layer's pre-swizzled weight image through a ring of shared-memory
//               stages with cp.async.bulk (mbarrier complete_tx); both slots consume a stage before it is refilled
//
// Tensor memory per slot (256 columns): X = residual stream (64), Z = layer output (64), A_hi / A_lo = next
// operand (64 + 64).  Residual additions never touch registers: the last layer of a DenseSkipBlock and proj2 of a
// gated block ACCUMULATE into X (alpha folded into the weights).  Biases ride in a constant-1 operand column;
// LayerNorm affine, SELU scale and the final rotation are folded into the weight images by pack_tc_kernel.
// Layers with separate ref / alt weights: proj1 computes both sets side by side in N and each row keeps its half;
// proj2 stacks both sets along K and each row feeds only its own half of the operand.
// The only cross-read coupling -- the per-variant mean fields of the gated blocks and the final set sums -- goes
// through a small shared exchange buffer between the four epilogue warps of a slot.
//
// Precision modes (pmt_set_precision): TF32 (one MMA per k-step; the tensor core truncates fp32 inputs to TF32)
// and TF32x3 (hi/lo split of both operands, Ahi.Bhi + Alo.Bhi + Ahi.Blo, ~2^-20 relative error: the fp32-parity
// mode).  Tiles are planned by plan_tiles_kernel (greedy packing of whole variants, one warp per claim) so that
// every role of every CTA knows its tile list up front.
#include <cstdlib>
#include <cstring>

#include "pmt_call.h"

namespace pmt {
namespace tc {

// Training recompute: operand columns [col0, col0 + NC) of `row`, rounded to TF32, into the step's panels (pmt_tc.cuh).
template <int NC>
__device__ __forceinline__ void save_operand(unsigned char* op, int row, int col0, const float* v) {
#pragma unroll
  for (int i = 0; i < NC / 4; ++i)
    *reinterpret_cast<float4*>(op + panel_off(row, col0 / 4 + i)) =
        make_float4(rna_tf32(v[4 * i]), rna_tf32(v[4 * i + 1]), rna_tf32(v[4 * i + 2]), rna_tf32(v[4 * i + 3]));
}

template <int PASSES, bool SAVE, bool LONG>
__global__ void __launch_bounds__(FWD_THREADS, 1)
reads_forward_tc_kernel(const __grid_constant__ PmtModelDesc D, const __grid_constant__ TcPlan TP, const __grid_constant__ TcArgs A,
                        int n_stages, int stage_bytes) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // carve (pmt_tc.cuh): [Shared][xch 2 slots][sums 2 slots][pair exchange][block scalars][HeadConstTc][step table] at
  // constant offsets from `sb`, then the weight ring (n_stages x stage_bytes) at sb + FWD_RING, 1024-aligned
  const unsigned raw = smem_addr(smem_raw);
  const unsigned sb = ((raw + FWD_RING + 1023u) & ~1023u) - FWD_RING;
  const unsigned ring = sb + FWD_RING;
  unsigned char* const p = smem_raw + (sb - raw);
  Shared* S = reinterpret_cast<Shared*>(p);
  float* blkc = reinterpret_cast<float*>(p + FWD_BLKC);
  HeadConstTc* HCT = reinterpret_cast<HeadConstTc*>(p + FWD_HEAD);
  HeadConst* HC = &HCT->h;
  constexpr unsigned SH_TB = offsetof(Shared, tb), TB_BYTES = sizeof(TileBuf);
  constexpr unsigned TB_IDX = offsetof(TileBuf, idx), TB_SRC = offsetof(TileBuf, src), TB_WORDS = offsetof(TileBuf, words),
                     TB_VAR = offsetof(TileBuf, var), TB_V0 = offsetof(TileBuf, v0), TB_NV = offsetof(TileBuf, nv),
                     TB_REF_PAD = offsetof(TileBuf, ref_pad), TB_LT = offsetof(TileBuf, lt), TB_M = offsetof(TileBuf, m);
  constexpr unsigned HC_H = FWD_HEAD + offsetof(HeadConstTc, h);

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const float* W = A.wflat;
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_addr(&S->bar_a[s]), 8); mbar_init(smem_addr(&S->bar_d[s]), 1);
      for (int b = 0; b < 2; ++b) { mbar_init(smem_addr(&S->meta_full[s][b]), 1); mbar_init(smem_addr(&S->meta_free[s][b]), 8); }
    }
    for (int i = 0; i < n_stages; ++i) { mbar_init(smem_addr(&S->wfull[i]), 1); mbar_init(smem_addr(&S->wfree[i]), 2); }
    fence_mbar_init();
    head_constants(D, W, HC);
    for (int e = 0; e < MAXE; ++e) HCT->inv_sigma[e] = e < D.d_feat ? 1.f / HC->sigma[e] : 0.f;
    for (int s = 0; s < TP.n_steps; ++s) p[FWD_STEPS + s] = (unsigned char)(TP.step[s].epi | TP.step[s].blk << 4);
    for (int k = 0; k < MAXK; ++k) {
      const bool on = k < D.n_clusters;
      HCT->inv_two_tau2[k] = on ? 1.f / HC->two_tau2[k] : 0.f;
      HCT->inv_sqrt2_sigma[k] = on ? 1.f / HC->sqrt2_sigma[k] : 0.f;
      for (int e = 0; e < MAXE; ++e) HCT->unit[k][e] = (on && e < D.d_feat) ? W[D.unit_ke + k * D.d_feat + e] : 0.f;
    }
  }
  for (int i = tid; i < D.n_blocks * BC_STRIDE; i += FWD_THREADS) {
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

  // tiles [tile_first, n_tiles) of the list (the training recompute walks the list in bounded ranges)
  static_assert(!(LONG && SAVE), "the long-set tiles are forward only");
  const int tile_first = SAVE ? A.tile_first : 0;
  const int n_tiles = LONG ? __ldg(A.lng.n_tiles) : (SAVE ? min(__ldg(A.tiles), A.tile_limit) - tile_first : __ldg(A.tiles));
  const int n_slots = 2 * gridDim.x;
  // every slot of the CTA runs the same number of rounds (an idle slot processes an empty tile)
  // tile t of round r: slot 0 of every CTA first, then slot 1 (a small batch spreads over the SMs before it doubles up)
  const int rounds = n_tiles > (int)blockIdx.x ? (n_tiles - (int)blockIdx.x + n_slots - 1) / n_slots : 0;   // rounds of slot 0 >= slot 1
  const int n_steps = TP.n_steps;
  const unsigned tmem_base = __shfl_sync(0xffffffffu, S->tmem_base, 0);
  const bool l0_lo = A.batch.reads_kind != PMT_READS_U8;   // decoded reads k/32 and bits are exact in TF32

  if (warp == META_WARP) {
    // ===================================== tile meta producer =====================================
    // Everything a tile's set-up needs from global memory -- which variants, their row ranges, the gather indices and the
    // compressed rows themselves -- is a chain of four dependent loads.  This warp walks the chain one round ahead of the
    // epilogue warps and leaves the result in shared memory, so neither the tile set-up nor the decode step waits for it.
    const int lane = tid & 31;
    const long long total_ref = __ldg(A.batch.ref_off + A.batch.n_variants);
    const bool u8_rows = A.batch.reads_kind == PMT_READS_U8 && D.read_row_bytes == 12;
    const int DIS = D.d_info + D.d_seq;
    for (int round = 0; round < rounds; ++round) {
      const int b = round & 1;
      const unsigned fparity = ((round >> 1) & 1) ^ 1;   // the first use of each buffer finds it free
      for (int slot = 0; slot < 2; ++slot) {
        TileBuf* TB = &S->tb[slot][b];
        mbar_wait(smem_addr(&S->meta_free[slot][b]), fparity);
        const int t = (int)blockIdx.x + slot * (int)gridDim.x + round * n_slots;
        int v0 = 0, nv = 0;
        long long r_base = 0, a_base = 0;
        int nr_tot = 0, na_tot = 0, ref_pad = 0;
        if (LONG) {
          // one tile = up to TILE rows of one side of one long set: a ref tile is "all ref rows" (ref_pad = TILE), an alt
          // tile "all alt rows" (ref_pad = 0), so the per-row code below and in the epilogue warps needs no other change
          int4 d0 = make_int4(-1, 0, 0, 0), d1 = make_int4(0, 0, 0, 0);
          if (t < n_tiles) {
            const int4* lp = reinterpret_cast<const int4*>(A.lng.tiles + t);
            d0 = __ldg(lp); d1 = __ldg(lp + 1);
          }
          nv = d0.x >= 0 ? 1 : 0;
          v0 = nv ? d0.x : 0;
          int set_ref = 0, set_alt = 0;
          if (nv) {
            const long long r0 = __ldg(A.batch.ref_off + v0), a0 = __ldg(A.batch.alt_off + v0);
            set_ref = (int)(__ldg(A.batch.ref_off + v0 + 1) - r0); set_alt = (int)(__ldg(A.batch.alt_off + v0 + 1) - a0);
            r_base = r0 + (d0.y == 0 ? d0.z : 0); a_base = a0 + (d0.y == 1 ? d0.z : 0);
            nr_tot = d0.y == 0 ? d0.w : 0; na_tot = d0.y == 1 ? d0.w : 0;
            ref_pad = d0.y == 0 ? TILE : 0;
          }
          if (lane == 0) {
            TB->v0 = v0; TB->nv = nv; TB->ref_pad = ref_pad; TB->var[0] = v0;
            TB->lt[0] = d1.y; TB->lt[1] = d1.x; TB->lt[2] = d1.z; TB->lt[3] = d1.w; TB->lt[4] = d0.y; TB->lt[5] = d0.w;
            TB->lt[6] = set_ref; TB->lt[7] = set_alt;
            TB->m.ref_start[0] = 0; TB->m.ref_cnt[0] = (unsigned char)nr_tot;
            TB->m.alt_start[0] = (unsigned char)(ref_pad & 127); TB->m.alt_cnt[0] = (unsigned char)na_tot;
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) TB->m.rowvar[q * 32 + lane] = (q * 32 + lane < nr_tot + na_tot) ? (unsigned char)0 : (unsigned char)255;
          if (nv && lane == 0 && A.out.info_seq_be) {
            const char* e = reinterpret_cast<const char*>(A.out.info_seq_be + (long long)v0 * DIS);
            prefetch_l2(e);
          }
        } else {
          if (t < n_tiles) { v0 = __ldg(A.tiles + 2 + 2 * (tile_first + t)); nv = __ldg(A.tiles + 3 + 2 * (tile_first + t)); }
          // The tile's variants: positions [v0, v0 + nv) of the planner's permutation (A.perm; NULL: the variants themselves,
          // as the training recompute and the backward need them).  Lane l holds variants l, l + 32, ...
          int var[4], rc[4], ac[4];
          long long r0[4], a0[4];
          int rsum = 0, asum = 0;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int j = k * 32 + lane;
            var[k] = 0; rc[k] = 0; ac[k] = 0; r0[k] = 0; a0[k] = 0;
            if (j < nv) {
              var[k] = A.perm ? __ldg(A.perm + v0 + j) : v0 + j;
              r0[k] = __ldg(A.batch.ref_off + var[k]); a0[k] = __ldg(A.batch.alt_off + var[k]);
              rc[k] = (int)(__ldg(A.batch.ref_off + var[k] + 1) - r0[k]); ac[k] = (int)(__ldg(A.batch.alt_off + var[k] + 1) - a0[k]);
              if (A.out.info_seq_be) {   // the concat step's embedding rows: towards L2
                const char* e = reinterpret_cast<const char*>(A.out.info_seq_be + (long long)var[k] * DIS);
                prefetch_l2(e);
                prefetch_l2(e + DIS * 4 - 4);
              }
            }
            rsum += rc[k]; asum += ac[k];
          }
          // row layout of the tile: the ref rows of its variants in list order, padding to a multiple of four, the alt rows
          int rs[4], as[4];
          {
            int rcar = 0, acar = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              int ri = rc[k], ai = ac[k];
#pragma unroll
              for (int o = 1; o < 32; o <<= 1) {
                const int tr = __shfl_up_sync(0xffffffffu, ri, o), ta = __shfl_up_sync(0xffffffffu, ai, o);
                if (lane >= o) { ri += tr; ai += ta; }
              }
              rs[k] = rcar + ri - rc[k]; as[k] = acar + ai - ac[k];
              rcar += __shfl_sync(0xffffffffu, ri, 31); acar += __shfl_sync(0xffffffffu, ai, 31);
            }
            nr_tot = rcar; na_tot = acar;
          }
          (void)rsum; (void)asum; (void)r_base; (void)a_base;
          ref_pad = (nr_tot + 3) & ~3;
          if (lane == 0) { TB->v0 = v0; TB->nv = nv; TB->ref_pad = ref_pad; }
          reinterpret_cast<unsigned*>(TB->m.rowvar)[lane] = 0xFFFFFFFFu;   // 255 = padding row
#pragma unroll
          for (int q = 0; q < 4; ++q) TB->idx[q * 32 + lane] = -1;
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int j = k * 32 + lane;
            if (j < nv) {
              const int rsj = rs[k], asj = ref_pad + as[k];
              TB->var[j] = var[k];
              TB->m.ref_start[j] = (unsigned char)rsj; TB->m.ref_cnt[j] = (unsigned char)rc[k];
              TB->m.alt_start[j] = (unsigned char)asj; TB->m.alt_cnt[j] = (unsigned char)ac[k];
              for (int i = 0; i < rc[k]; ++i) { TB->m.rowvar[rsj + i] = (unsigned char)j; TB->idx[rsj + i] = r0[k] + i; }
              for (int i = 0; i < ac[k]; ++i) { TB->m.rowvar[asj + i] = (unsigned char)j; TB->idx[asj + i] = total_ref + a0[k] + i; }
            }
          }
        }
        __syncwarp();
        long long idx[4], src[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = q * 32 + lane;
          if (LONG) {
            idx[q] = -1;
            if (r < nr_tot) idx[q] = r_base + r;
            else if (r >= ref_pad && r - ref_pad < na_tot) idx[q] = total_ref + a_base + (r - ref_pad);
          } else {
            idx[q] = TB->idx[r];
          }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) src[q] = (idx[q] >= 0 && A.batch.read_indices) ? __ldg(A.batch.read_indices + idx[q]) : idx[q];
        unsigned w[4][3];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          w[q][0] = w[q][1] = w[q][2] = 0u;
          if (u8_rows && src[q] >= 0) {
            const unsigned* wp = reinterpret_cast<const unsigned*>(reinterpret_cast<const unsigned char*>(A.batch.reads) + src[q] * 12);
            w[q][0] = __ldg(wp); w[q][1] = __ldg(wp + 1); w[q][2] = __ldg(wp + 2);
          }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = q * 32 + lane;
          TB->idx[r] = idx[q]; TB->src[r] = src[q];
          TB->words[r * 3] = w[q][0]; TB->words[r * 3 + 1] = w[q][1]; TB->words[r * 3 + 2] = w[q][2];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_addr(&S->meta_full[slot][b]));   // release semantics: the stores above are visible
      }
    }
  } else if (warp == LOAD_WARP) {
    // ===================================== weight loader =====================================
    if (elect_one()) {
      const long long total = (long long)rounds * n_steps;
      int stage = 0, step = 0;
      unsigned parity = 1;   // first pass through the ring: stages are free
      for (long long g = 0; g < total; ++g) {
        mbar_wait(smem_addr(&S->wfree[stage]), parity);
        const TcStep& o = TP.step[step];
        const unsigned bytes = o.img_bytes * (PASSES == 3 ? 2 : 1);
        mbar_expect_tx(smem_addr(&S->wfull[stage]), bytes);
        bulk_g2s(ring + stage * stage_bytes, A.image + o.img_off, bytes, smem_addr(&S->wfull[stage]));
        if (++stage == n_stages) { stage = 0; parity ^= 1; }
        if (++step == n_steps) step = 0;
      }
    }
    __syncwarp();
  } else if (warp >= MMA_WARP) {
    // ===================================== MMA issuers: one warp per slot =====================================
    // Each warp blocks only on ITS slot's operand barrier, so the two slots drift apart freely and one slot's
    // MMA overlaps the other slot's epilogue; a weight stage is released when both warps have committed past it.
    const int s = warp - MMA_WARP;
    const unsigned tb = tmem_base + s * SLOT_COLS;
    const unsigned bar_a = smem_addr(&S->bar_a[s]), bar_d = smem_addr(&S->bar_d[s]);
    int stage = 0;
    unsigned wparity = 0, aparity = 0;
    for (int round = 0; round < rounds; ++round) {
      for (int step = 0; step < n_steps; ++step) {
        const TcStep& o = TP.step[step];
        const int oN = o.N, oKS = o.KS, o_dst_x = o.dst_x, o_img_bytes = o.img_bytes;
        const unsigned idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(oN >> 3) << 17) | ((128u >> 4) << 24);
        const unsigned wb = ring + stage * stage_bytes;
        const uint64_t b_hi = smem_desc(wb), b_lo = smem_desc(wb + o_img_bytes);
        const unsigned kb_stride16 = (unsigned)(oN * 128) >> 4;
        const bool lo_pass = step > 0 || l0_lo;
        const unsigned d = tb + (o_dst_x ? COL_X : COL_Z);
        mbar_wait(smem_addr(&S->wfull[stage]), wparity);
        mbar_wait(bar_a, aparity);
        tc_fence_after();
        if (elect_one()) {
          switch (oKS) {
            case 3: issue_chain<3, PASSES>(d, tb + COL_AHI, tb + COL_ALO, b_hi, b_lo, kb_stride16, idesc, o_dst_x, lo_pass); break;
            case 4: issue_chain<4, PASSES>(d, tb + COL_AHI, tb + COL_ALO, b_hi, b_lo, kb_stride16, idesc, o_dst_x, lo_pass); break;
            default: issue_chain<8, PASSES>(d, tb + COL_AHI, tb + COL_ALO, b_hi, b_lo, kb_stride16, idesc, o_dst_x, lo_pass); break;
          }
          mma_commit(bar_d);
          mma_commit(smem_addr(&S->wfree[stage]));
        }
        __syncwarp();
        aparity ^= 1;
        if (++stage == n_stages) { stage = 0; wparity ^= 1; }
      }
    }
  } else {
    // ============ epilogue: two threads per row; thread (row, half) owns 32 of the row's 64 columns ============
    const int slot = warp >> 3, half = (warp >> 2) & 1, quarter = warp & 3;
    const int lane = tid & 31;
    const int row = quarter * 32 + lane;
    const int srow = half * TILE + row;              // 0..255 inside the slot
    const int slot_bar = 1 + slot, pair_bar = 3 + slot * 4 + quarter;
    const unsigned xch = sb + FWD_XCH + slot * XCH_ROWS * XCH_LD * 4;    // [XCH_ROWS][XCH_LD] floats
    const unsigned sums = sb + FWD_SUMS + slot * SUMS_FLOATS * 4;        // [segment = 2 * variant + side][MAXH]
    const unsigned px_mine = sb + FWD_PAIRX + ((slot * 2 + half) * TILE + row) * 8, px_other = sb + FWD_PAIRX + ((slot * 2 + (half ^ 1)) * TILE + row) * 8;
    const unsigned bar_a = sb + offsetof(Shared, bar_a) + slot * 8, bar_d = sb + offsetof(Shared, bar_d) + slot * 8;
    const unsigned steps = sb + FWD_STEPS;
    const unsigned trow = tmem_base + slot * SLOT_COLS + ((unsigned)(quarter * 32) << 16);
    const unsigned t_x = trow + COL_X, t_z = trow + COL_Z, t_hi = trow + COL_AHI, t_lo = trow + COL_ALO;
    const int E = D.d_feat, K = D.n_clusters, Dm = D.d_model, H = D.d_ffn / 2, DR = D.d_read, F = D.n_read_features;
    const int DIS = D.d_info + D.d_seq;
    const int B = A.batch.n_variants;
    const long long total_ref = __ldg(A.batch.ref_off + B);
    const unsigned inv_h = (65536u + (unsigned)H - 1u) / (unsigned)H, inv_e = (65536u + (unsigned)E - 1u) / (unsigned)E;
    const int n_half = half ? DIS : DR;              // real columns of this thread's half of a d_model vector
    unsigned dparity = 0;

    for (int round = 0; round < rounds; ++round) {
      const int t = (int)blockIdx.x + slot * (int)gridDim.x + round * n_slots;
      // ---------------- tile meta: prepared by the meta warp while the previous tile was computed ----------------
      const unsigned tb = sb + SH_TB + (slot * 2 + (round & 1)) * TB_BYTES;   // this round's TileBuf
      const unsigned m_rowvar = tb + TB_M + offsetof(SlotMeta, rowvar), m_ref_start = tb + TB_M + offsetof(SlotMeta, ref_start),
                     m_ref_cnt = tb + TB_M + offsetof(SlotMeta, ref_cnt), m_alt_start = tb + TB_M + offsetof(SlotMeta, alt_start),
                     m_alt_cnt = tb + TB_M + offsetof(SlotMeta, alt_cnt), tb_var = tb + TB_VAR;
      mbar_wait(sb + offsetof(Shared, meta_full) + (slot * 2 + (round & 1)) * 8, (round >> 1) & 1);
      const int v0 = lds_s32(tb + TB_V0), nv = lds_s32(tb + TB_NV), ref_pad = lds_s32(tb + TB_REF_PAD);
      const int lt_first = LONG ? lds_s32(tb + TB_LT) : 0, lt_k = LONG ? lds_s32(tb + TB_LT + 4) : 0, lt_tref = LONG ? lds_s32(tb + TB_LT + 8) : 0,
                lt_talt = LONG ? lds_s32(tb + TB_LT + 12) : 0, lt_side = LONG ? lds_s32(tb + TB_LT + 16) : 0, lt_rows = LONG ? lds_s32(tb + TB_LT + 20) : 0,
                set_ref = LONG ? lds_s32(tb + TB_LT + 24) : 0, set_alt = LONG ? lds_s32(tb + TB_LT + 28) : 0;
      const long long my_idx = lds_s64(tb + TB_IDX + row * 8), my_src = lds_s64(tb + TB_SRC + row * 8);
      unsigned char* const scr = (SAVE && t < n_tiles) ? A.scratch + (size_t)t * TP.tile_bytes : nullptr;
      const int rv = (int)lds_u8(m_rowvar + row);
      const int my_var = rv == 255 ? -1 : rv;
      const bool is_alt = row >= ref_pad;

      // step kind and gated block (epi | blk << 4): the next step's entry is read before the accumulator wait
      unsigned code = lds_u8(steps);
      for (int step = 0; step < n_steps; ++step) {
        const int epi = (int)(code & 15u), blk = (int)(code >> 4);
        unsigned char* const scr_op = (SAVE && scr) ? scr + TP.step[step].scr_off : nullptr;
        switch (epi) {
          case EPI_DECODE: {   // batch.py:51-56, plain_text_data.py:510-511 (quirk Q2: the uint8 de-quantisation wraps)
            float v[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = 0.f;
            if (my_idx >= 0) {
              const long long src = my_src;
              if (A.batch.reads_kind == PMT_READS_U8) {
                const int rb = D.read_row_bytes;
                const unsigned char* rp = reinterpret_cast<const unsigned char*>(A.batch.reads) + src * rb;
                unsigned bytes[8];   // this half's 8 source bytes: packed bytes 0..3, or packed bytes 4..6 + quantised 7..
                if (rb == 12) {      // the meta warp fetched the row
                  if (half == 0) {
                    const unsigned w0 = (unsigned)lds_s32(tb + TB_WORDS + row * 12);
#pragma unroll
                    for (int b = 0; b < 4; ++b) bytes[b] = (w0 >> (8 * b)) & 255u;
                  } else {
                    const unsigned w1 = (unsigned)lds_s32(tb + TB_WORDS + row * 12 + 4), w2 = (unsigned)lds_s32(tb + TB_WORDS + row * 12 + 8);
#pragma unroll
                    for (int b = 0; b < 4; ++b) { bytes[b] = (w1 >> (8 * b)) & 255u; bytes[4 + b] = (w2 >> (8 * b)) & 255u; }
                  }
                } else {
#pragma unroll
                  for (int b = 0; b < 8; ++b) {
                    const int sb = half * 4 + b;
                    bytes[b] = (sb < rb && (half == 1 || b < 4)) ? (unsigned)__ldg(rp + sb) : 128u;
                  }
                }
                if (half == 0) {
#pragma unroll
                  for (int b = 0; b < 4; ++b)
#pragma unroll
                    for (int bit = 0; bit < 8; ++bit) v[b * 8 + bit] = __uint_as_float((0u - ((bytes[b] >> (7 - bit)) & 1u)) & 0x3f800000u);
                } else {
#pragma unroll
                  for (int b = 0; b < 3; ++b)
#pragma unroll
                    for (int bit = 0; bit < 8; ++bit) v[b * 8 + bit] = __uint_as_float((0u - ((bytes[b] >> (7 - bit)) & 1u)) & 0x3f800000u);
                  if (rb == 12) {
#pragma unroll
                    for (int b = 3; b < 8; ++b) v[24 + b - 3] = (float)((bytes[b] + 128u) & 255u) * 0.03125f;
                  } else {
#pragma unroll
                    for (int b = 3; b < 8; ++b)
                      if (4 + b < rb) v[24 + b - 3] = (float)((bytes[b] + 128u) & 255u) * 0.03125f;
                  }
                }
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                  const int f = half * 32 + i;
                  if (f < F)
                    v[i] = A.batch.reads_kind == PMT_READS_F16 ? __half2float(reinterpret_cast<const __half*>(A.batch.reads)[src * F + f])
                                                               : reinterpret_cast<const float*>(A.batch.reads)[src * F + f];
                }
              }
            }
            if (half == 1) v[31] = 1.f;   // operand column 63: bias
            if (SAVE && scr_op) save_operand<32>(scr_op, row, half * 32, v);
            store_operand<32, PASSES>(t_hi + half * 32, t_lo + half * 32, v, l0_lo);
          } break;
          case EPI_FIRST32: {   // mlp.py:61-62 then the first DenseSkipBlock's leading SELU (mlp.py:8-22)
            float v[16];
            load_cols<16>(t_z + half * 16, v);
            unsigned r[16];
            selu_u_n<16>(v);
#pragma unroll
            for (int i = 0; i < 16; i += 2) {
              up2(mul2(pk2(v[i], v[i + 1]), pk2(SELU_SCALE, SELU_SCALE)), v[i], v[i + 1]);
              r[i] = __float_as_uint(v[i]); r[i + 1] = __float_as_uint(v[i + 1]);
            }
            tmem_st16(t_x + half * 16, r);
            if (SAVE && scr) {
              float* x0 = reinterpret_cast<float*>(scr + TP.x0_off) + (half * 16) * TILE + row;
#pragma unroll
              for (int i = 0; i < 16; ++i) x0[i * TILE] = v[i];
            }
            selu_u_n<16>(v);
            if (half == 1) v[15] = 1.f;   // operand column 31: bias
            if (SAVE && scr_op) save_operand<16>(scr_op, row, half * 16, v);
            store_operand<16, PASSES>(t_hi + half * 16, t_lo + half * 16, v, true);
          } break;
          case EPI_ACT_Z32:
          case EPI_ACT_X32: {
            float v[16];
            load_cols<16>((epi == EPI_ACT_Z32 ? t_z : t_x) + half * 16, v);
            selu_u_n<16>(v);
            if (half == 1) v[15] = 1.f;
            if (SAVE && scr_op) save_operand<16>(scr_op, row, half * 16, v);
            store_operand<16, PASSES>(t_hi + half * 16, t_lo + half * 16, v, true);
          } break;
          case EPI_LN_FIRST:
          case EPI_LN: {   // gated_mlp.py:185 (LayerNorm affine folded into proj1); artifact_model.py:246-251 concat
            float v[32];
            if (epi == EPI_LN_FIRST && half == 1) {
              const float* src = my_var >= 0 ? A.out.info_seq_be + (long long)lds_s32(tb_var + my_var * 4) * DIS : nullptr;
              unsigned r[32];
#pragma unroll
              for (int i = 0; i < 32; ++i) { v[i] = (src && i < DIS) ? __ldg(src + i) : 0.f; r[i] = __float_as_uint(v[i]); }
              tmem_st32(t_x + 32, r);
            } else {
              load_cols<32>(t_x + half * 32, v);
            }
            // statistics of this half (padding columns are zero), combined with the partner's (Chan et al.)
            const float nh = (float)n_half, no = (float)(Dm - n_half);
            const float s_h = sum_n<32>(v);
            const float m_h = s_h / nh;
            const float q_h = sumsq_centered_n<32>(v, m_h) - (32.f - nh) * m_h * m_h;
            sts_f32x2(px_mine, s_h, q_h);
            named_barrier(pair_bar, 64);
            const float2 oth = lds_f32x2(px_other);
            const float mean = (s_h + oth.x) / (float)Dm;
            const float dm = m_h - oth.x / no;
            const float var = (q_h + oth.y + dm * dm * nh * no / (float)Dm) / (float)Dm;
            const float rstd = rsqrtf(fmaxf(var, 0.f) + LN_EPS);
            const float shift = -mean * rstd;
            {
              const f32x2 rs2 = pk2(rstd, rstd), sh2 = pk2(shift, shift);
#pragma unroll
              for (int i = 0; i < 32; i += 2) up2(fma2(pk2(v[i], v[i + 1]), rs2, sh2), v[i], v[i + 1]);
            }
            if (half == 0) v[31] = 1.f;   // operand column 31: bias
            if (SAVE && scr_op) {
              save_operand<32>(scr_op, row, half * 32, v);
              if (half == 0) reinterpret_cast<float*>(scr + TP.rstd_off)[blk * TILE + row] = rstd;
            }
            store_operand<32, PASSES>(t_hi + half * 32, t_lo + half * 32, v, true);
          } break;
          case EPI_GATE: {   // gated_mlp.py:186-190, 228-251; this thread gates hidden units [k0, k0 + 6)
            const unsigned bcs = sb + FWD_BLKC + blk * BC_STRIDE * 4;
            // proj1 output: [ref set | alt set], one set = [z1 at 0..H) | z2 at 12..12+H)]
            float z1s[16], z2s[16];
            {
              unsigned r1[16], r2[16];
              const unsigned base = t_z + (is_alt ? NP1 : 0);
              // addresses must be warp-uniform: load both sets when the warp mixes ref and alt rows
              const bool all_ref = __all_sync(0xffffffffu, !is_alt), all_alt = __all_sync(0xffffffffu, is_alt);
              if (all_ref || all_alt) {
                const unsigned ub = t_z + (all_alt ? NP1 : 0);
                tmem_ld8(ub + half * 6, r1); tmem_ld16(ub + NP1 / 2, r2);
                tmem_wait_ld();
              } else {
                unsigned a1[8], a2[16];
                tmem_ld8(t_z + half * 6, r1); tmem_ld16(t_z + NP1 / 2, r2);
                tmem_ld8(t_z + NP1 + half * 6, a1); tmem_ld16(t_z + NP1 + NP1 / 2, a2);
                tmem_wait_ld();
#pragma unroll
                for (int i = 0; i < 8; ++i) r1[i] = is_alt ? a1[i] : r1[i];
#pragma unroll
                for (int i = 0; i < 16; ++i) r2[i] = is_alt ? a2[i] : r2[i];
              }
              (void)base;
#pragma unroll
              for (int i = 0; i < 8; ++i) z1s[i] = __uint_as_float(r1[i]);
#pragma unroll
              for (int i = 0; i < 16; ++i) z2s[i] = __uint_as_float(r2[i]);
            }
            // z1s[j] = z1[k0 + j] (j < 6), z2s[k] = z2[k] (k < 12; columns >= H are zero)
            const int k0 = half * 6;
            float z2[12];
            selu_u_n<12>(z2s);
#pragma unroll
            for (int k = 0; k < 12; k += 2) {
              float s0, s1;
              up2(mul2(pk2(z2s[k], z2s[k + 1]), pk2(SELU_SCALE, SELU_SCALE)), s0, s1);
              z2[k] = k < H ? s0 : 0.f; z2[k + 1] = k + 1 < H ? s1 : 0.f;
            }
            const float mean = sum_n<12>(z2) / (float)H;
            float var;
            {
              float a0 = 0.f, a1 = 0.f;
#pragma unroll
              for (int k = 0; k < 12; k += 2) {
                const float d0 = k < H ? z2[k] - mean : 0.f, d1 = k + 1 < H ? z2[k + 1] - mean : 0.f;
                a0 = fmaf(d0, d0, a0); a1 = fmaf(d1, d1, a1);
              }
              var = (a0 + a1) / (float)H;
            }
            const float rstd = rsqrtf(var + LN_EPS);
            float z2n[6];
#pragma unroll
            for (int j = 0; j < 6; ++j) {
              // z2[k0 + j]: k0 is 0 or 6 -> select between two compile-time registers
              const float zz = half ? z2[j + 6] : z2[j];
              z2n[j] = (zz - mean) * rstd * lds_f32(bcs + (BC_LN2W + k0 + j) * 4) + lds_f32(bcs + (BC_LN2B + k0 + j) * 4);
              if (k0 + j < H) sts_f32(xch + ((k0 + j) * XCH_LD + row) * 4, z2n[j]);
              if (SAVE && scr) {   // what the backward of the gate needs: xhat2, selu'(z2), (z1 below), 1 / std
                float* gi = reinterpret_cast<float*>(scr + TP.gate_off) + ((blk * GATE_ITEMS) * 2 + half) * TILE + row;
                gi[(6 + j) * 2 * TILE] = (zz - mean) * rstd;
                gi[(12 + j) * 2 * TILE] = zz > 0.f ? SELU_SCALE : zz + SELU_SCALE * SELU_ALPHA;
                if (j == 0) gi[18 * 2 * TILE] = rstd;
              }
            }
            // the z1 activations do not depend on the other rows: computed while the slower warps reach the barrier
            float z1a[6];
            selu_u_n<6>(z1s);
#pragma unroll
            for (int j = 0; j < 6; j += 2) up2(mul2(pk2(z1s[j], z1s[j + 1]), pk2(SELU_SCALE, SELU_SCALE)), z1a[j], z1a[j + 1]);
            named_barrier(slot_bar, 256);
            if (LONG) {   // mean fields of a set spread over many tiles (pmt_tc.cuh: LongTile)
              const float regw = lds_f32(bcs + BC_REGW * 4);
              const int nb = D.n_blocks;
              // (a) column sums of this tile's rows -> the tile's slot in global memory; a lane pair per hidden unit
              if (srow < 32) {
                const int f = lane >> 1, part = lane & 1;
                const bool on = f < H && nv > 0;
                const unsigned src = xch + ((on ? f : 0) * XCH_LD + part) * 4;
                const int mine = on ? (lt_rows - part + 1) >> 1 : 0;
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
                for (int i = 0; i < mine; i += 4) {
                  const float x0 = lds_f32(src + i * 8), x1 = lds_f32(src + i * 8 + 8), x2 = lds_f32(src + i * 8 + 16), x3 = lds_f32(src + i * 8 + 24);
                  a0 += x0;
                  a1 += i + 1 < mine ? x1 : 0.f;
                  a2 += i + 2 < mine ? x2 : 0.f;
                  a3 += i + 3 < mine ? x3 : 0.f;
                }
                float acc = (a0 + a1) + (a2 + a3);
                acc += __shfl_xor_sync(0xffffffffu, acc, 1);
                if (on && part == 0) A.lng.mf_part[((size_t)(lt_first + lt_k) * nb + blk) * MAXH + f] = acc;
                __threadfence();
                __syncwarp();
                // (b) arrive, then wait for the set's other tiles (all in flight: the list never lets a set straddle a round)
                if (lane == 0 && nv > 0) {
                  int* c = A.lng.mf_cnt + (size_t)lt_first * nb + blk;
                  atomicAdd(c, 1);
                  const int T = lt_tref + lt_talt;
                  while (ld_acquire_gpu(c) < T) __nanosleep(20);
                  __threadfence();
                }
                __syncwarp();
                // (c) totals in tile order -> the slot's mean-field table (segment 0 = ref, 1 = alt)
                if (lane < 2 * MAXH && nv > 0) {
                  const int s = lane >= MAXH ? 1 : 0, ff = lane - s * MAXH;
                  if (ff < H) {
                    const int t0 = s ? lt_tref : 0, tn = s ? lt_talt : lt_tref;
                    float tot = 0.f;
                    for (int tt = 0; tt < tn; ++tt) tot += __ldcg(A.lng.mf_part + ((size_t)(lt_first + t0 + tt) * nb + blk) * MAXH + ff);
                    const float num = s == 0 ? tot + regw * lds_f32(bcs + (BC_REG + ff) * 4) : tot;
                    const float den = s == 0 ? (float)set_ref + regw : (float)set_alt + 1e-4f;
                    sts_f32(sums + (s * MAXH + ff) * 4, __fdividef(num, den));
                  }
                }
              }
            } else {   // per-variant mean fields (gated_mlp.py:236-239)
              // two threads (a lane pair) per sum: even / odd rows of the set, combined with one shuffle
              const float regw = lds_f32(bcs + BC_REGW * 4);
              const int n_sums = nv * 2 * H;
              const int part = lane & 1;
              for (int base = (srow >> 1) & ~15; base < n_sums; base += 128) {
                const int idx = base + (lane >> 1);
                const bool on = idx < n_sums;
                const int seg = on ? (int)(((unsigned)idx * inv_h) >> 16) : 0, f = on ? idx - seg * H : 0;
                const int j = seg >> 1, s = seg & 1;
                const int start = (int)lds_u8((s ? m_alt_start : m_ref_start) + j);
                const int cnt = on ? (int)lds_u8((s ? m_alt_cnt : m_ref_cnt) + j) : 0;
                const unsigned src = xch + (f * XCH_LD + start + part) * 4;
                // this thread's rows: part, part + 2, ...; four independent loads per trip (the tail reads inside the exchange
                // buffer and is masked): the trip count of a warp is that of its longest set
                const int mine = (cnt - part + 1) >> 1;
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
                for (int i = 0; i < mine; i += 4) {
                  const float x0 = lds_f32(src + i * 8), x1 = lds_f32(src + i * 8 + 8), x2 = lds_f32(src + i * 8 + 16), x3 = lds_f32(src + i * 8 + 24);
                  a0 += x0;
                  a1 += i + 1 < mine ? x1 : 0.f;
                  a2 += i + 2 < mine ? x2 : 0.f;
                  a3 += i + 3 < mine ? x3 : 0.f;
                }
                float acc = (a0 + a1) + (a2 + a3);
                acc += __shfl_xor_sync(0xffffffffu, acc, 1);
                if (on && part == 0) {
                  const float num = s == 0 ? acc + regw * lds_f32(bcs + (BC_REG + f) * 4) : acc;
                  const float den = (float)cnt + (s == 0 ? regw : 1e-4f);
                  const float m = __fdividef(num, den);
                  sts_f32(sums + (seg * MAXH + f) * 4, m);
                  if (SAVE && scr) reinterpret_cast<float*>(scr + TP.means_off)[(blk * 2 * BWD_MAXV + seg) * MAXH + f] = m;
                }
              }
            }
            named_barrier(slot_bar, 256);
            // proj2 operand columns of this thread: [t_ref (6) | t_alt (6)]; the second thread's last two hidden
            // slots (k = 10 would be unit 11; MAXH = 11 -> slot 5 of half 1 is unit 11 < MAXH only if H = 11)
            // layout, half 0: [t_ref k 0..5 | t_alt k 0..5]; half 1: [t_ref k 6..10 | t_alt k 6..10 | is_ref, is_alt]
            float v[12];
            {
              const float alpha = lds_f32(bcs + (is_alt ? BC_AALT : BC_AREF) * 4);
              const float beta = lds_f32(bcs + (is_alt ? BC_BALT : BC_BREF) * 4);
              const float gamma = is_alt ? lds_f32(bcs + BC_GAMMA * 4) : 0.f;
              const int mv = my_var >= 0 ? my_var : 0;
              const unsigned s_ref = sums + ((mv * 2 + 0) * MAXH + k0) * 4, s_own = sums + ((mv * 2 + (is_alt ? 1 : 0)) * MAXH + k0) * 4;
              float tk[6];
#pragma unroll
              for (int j = 0; j < 6; ++j) {
                tk[j] = 0.f;
                if (k0 + j < H) {
                  float gate = fmaf(z2n[j], alpha, 1.f);
                  if (my_var >= 0) {
                    const float m_ref = lds_f32(s_ref + j * 4), m_own = lds_f32(s_own + j * 4);
                    gate = fmaf(beta, m_own, fmaf(gamma, m_ref, gate));
                  }
                  const float z1 = z1a[j];
                  tk[j] = z1 * gate;
                  if (SAVE && scr)
                    reinterpret_cast<float*>(scr + TP.gate_off)[((blk * GATE_ITEMS + j) * 2 + half) * TILE + row] = z1;
                }
              }
              if (half == 0) {
#pragma unroll
                for (int j = 0; j < 6; ++j) { v[j] = is_alt ? 0.f : tk[j]; v[6 + j] = is_alt ? tk[j] : 0.f; }
              } else {
#pragma unroll
                for (int j = 0; j < 5; ++j) { v[j] = is_alt ? 0.f : tk[j]; v[5 + j] = is_alt ? tk[j] : 0.f; }
                v[10] = is_alt ? 0.f : 1.f;
                v[11] = is_alt ? 1.f : 0.f;
              }
            }
            if (SAVE && scr_op) save_operand<12>(scr_op, row, half * 12, v);
            store_operand<12, PASSES>(t_hi + half * 12, t_lo + half * 12, v, true);
          } break;
          case EPI_ACT_X64:
          case EPI_ACT_Z64:
          case EPI_COPY_X64: {
            float v[32];
            load_cols<32>((epi == EPI_ACT_Z64 ? t_z : t_x) + half * 32, v);
            if (epi != EPI_COPY_X64) selu_u_n<32>(v);
            if (half == 0) v[31] = 1.f;
            if (SAVE && scr_op) save_operand<32>(scr_op, row, half * 32, v);
            store_operand<32, PASSES>(t_hi + half * 32, t_lo + half * 32, v, true);
          } break;
        }
        // ---- hand the operand to the MMA warp, wait for the accumulator ----
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_a);
        code = lds_u8(steps + (step + 1 < n_steps ? step + 1 : 0));
        mbar_wait(bar_d, dparity);
        dparity ^= 1;
        tc_fence_after();
      }

      // ---------------- clustering head (rotation folded into the last layer; feature_clustering.py:82-135) ----------------
      // Both threads of a row hold its features.  half 0: feature rows for the set means, the non-artifact term and the
      // even clusters; half 1: the outlier term and the odd clusters.
      float f[MAXE];
      load_cols<MAXE>(t_z, f);
      if (half == 0) {
#pragma unroll
        for (int i = 0; i < MAXE; ++i) if (i < E) sts_f32(xch + (i * XCH_LD + row) * 4, f[i]);
        if (A.out.final_re && my_idx >= 0) {
#pragma unroll
          for (int e = 0; e < MAXE; ++e) if (e < E) A.out.final_re[my_idx * E + e] = f[e];
        }
        if (SAVE && scr) {
          float* fo = reinterpret_cast<float*>(scr + TP.f_off) + row;
#pragma unroll
          for (int e = 0; e < MAXE; ++e) fo[e * TILE] = e < E ? f[e] : 0.f;
        }
      }
      if (is_alt && my_var >= 0) {
        {   // (f / (2 sigma))^2 == (f / sigma)^2 / 4 exactly: one sum serves the non-artifact and the outlier Gaussians
          float q = 0.f;
#pragma unroll
          for (int e = 0; e < MAXE; ++e) { const float a = f[e] * lds_f32(sb + FWD_HEAD + offsetof(HeadConstTc, inv_sigma) + e * 4); q = fmaf(a, a, q); }
          const float c_ = lds_f32(sb + HC_H + (half ? offsetof(HeadConst, c_out) : offsetof(HeadConst, c_non)));
          sts_f32(xch + ((MAXE + half) * XCH_LD + row) * 4, half ? c_ - q * 0.125f : c_ - q * 0.5f);
        }
        for (int k = half; k < K; k += 2) {
          const unsigned u = sb + FWD_HEAD + offsetof(HeadConstTc, unit) + k * MAXE * 4, hk = sb + HC_H + k * 4;
          float pr = 0.f;
#pragma unroll
          for (int e = 0; e < MAXE; ++e) pr = fmaf(f[e], lds_f32(u + e * 4), pr);
          float o2 = 0.f;
#pragma unroll
          for (int e = 0; e < MAXE; ++e) { const float dd = fmaf(-pr, lds_f32(u + e * 4), f[e]); o2 = fmaf(dd, dd, o2); }
          const float dist = sqrtf(o2);
          const float ll_orth = lds_f32(hk + offsetof(HeadConst, c_orth)) -
                                (dist * dist) * lds_f32(sb + FWD_HEAD + offsetof(HeadConstTc, inv_two_tau2) + k * 4);
          const float ll_par = lds_f32(hk + offsetof(HeadConst, log_half_lambda)) +
                               logerfc((lds_f32(hk + offsetof(HeadConst, shift)) - pr) * lds_f32(sb + FWD_HEAD + offsetof(HeadConstTc, inv_sqrt2_sigma) + k * 4)) +
                               lds_f32(hk + offsetof(HeadConst, half_lambda)) * (lds_f32(hk + offsetof(HeadConst, two_mu_plus)) - 2.f * pr);
          sts_f32(xch + ((MAXE + 2 + k) * XCH_LD + row) * 4, ll_orth + ll_par);
        }
      }
      named_barrier(slot_bar, 256);
      // ---- per-variant sums and outputs (ragged_sets.py:144-158; artifact_model.py:291-292) ----
      if (LONG) {
        // This tile's raw sums (features of its side; for an alt tile also the K + 2 log-likelihood terms) go to its slot of
        // fin_part; the tile that arrives last adds the set's partials up in tile order and writes the set's outputs.
        float* fp = A.lng.fin_part + (size_t)(lt_first + lt_k) * LONG_FIN_W;
        const int n_items = nv > 0 ? E + (lt_side ? K + 2 : 0) : 0;
        {   // four threads per sum (rows i, i + 4, ...), combined with two shuffles; groups of four lanes stay inside a warp
          const int item = srow >> 2, part = srow & 3;
          const bool on = item < n_items;
          const int xr = item < E ? item : MAXE + (item - E);
          const unsigned src = xch + ((on ? xr : 0) * XCH_LD + part) * 4;
          const int mine = on ? (lt_rows - part + 3) >> 2 : 0;
          float a0 = 0.f, a1 = 0.f;
          for (int i = 0; i < mine; i += 2) {
            const float x0 = lds_f32(src + i * 16), x1 = lds_f32(src + i * 16 + 16);
            a0 += x0;
            a1 += i + 1 < mine ? x1 : 0.f;
          }
          float acc = a0 + a1;
          acc += __shfl_xor_sync(0xffffffffu, acc, 1);
          acc += __shfl_xor_sync(0xffffffffu, acc, 2);
          if (on && part == 0) fp[xr] = acc;
        }
        __threadfence();
        named_barrier(slot_bar, 256);
        if (srow < 32) {
          int last = 0;
          if (lane == 0 && nv > 0) {
            __threadfence();
            last = atomicAdd(A.lng.fin_cnt + lt_first, 1) == lt_tref + lt_talt - 1 ? 1 : 0;
            if (last) __threadfence();
          }
          last = __shfl_sync(0xffffffffu, last, 0);
          if (last) {
            const float* base = A.lng.fin_part + (size_t)lt_first * LONG_FIN_W;
            // set means (ragged_sets.py:144-158): lane = feature, both sides
            for (int s2 = 0; s2 < 2; ++s2) {
              float* dst = s2 ? A.out.alt_means_be : A.out.ref_means_be;
              const int t0 = s2 ? lt_tref : 0, tn = s2 ? lt_talt : lt_tref;
              if (dst && lane < E) {
                float tot = 0.f;
                for (int tt = 0; tt < tn; ++tt) tot += __ldcg(base + (size_t)(t0 + tt) * LONG_FIN_W + lane);
                dst[(long long)v0 * E + lane] = __fdividef(tot, (float)(s2 ? set_alt : set_ref) + 1e-4f);
              }
            }
            // log-likelihood sums over the alt reads (feature_clustering.py:82-135): lane = term
            const int k = lane;
            const bool term = k < K + 2;
            float acc = 0.f;
            if (term) {
              for (int tt = 0; tt < lt_talt; ++tt) acc += __ldcg(base + (size_t)(lt_tref + tt) * LONG_FIN_W + MAXE + k);
              if (k >= 2) acc += lds_f32(sb + HC_H + offsetof(HeadConst, logw) + (k - 2) * 4);
            }
            const bool art_term = term && k >= 2;
            float art_max = art_term ? acc : -INFINITY;
#pragma unroll
            for (int m = 1; m < 8; m <<= 1) art_max = fmaxf(art_max, __shfl_xor_sync(0xffffffffu, art_max, m));
            float sacc = art_term ? expf(acc - art_max) : 0.f;
#pragma unroll
            for (int m = 1; m < 8; m <<= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, m);
            const float ll0 = __shfl_sync(0xffffffffu, acc, 0), ll1 = __shfl_sync(0xffffffffu, acc, 1);
            if (term) {
              const long long v = v0;
              const float art = art_max + logf(sacc);
              if (A.out.logits_bk) A.out.logits_bk[v * (K + 2) + k] = acc;
              if (k == 0 && A.out.logits_b) A.out.logits_b[v] = 20.f * tanhf((art - ll0) / 20.f);
              if (k == 1 && A.out.outlier_logits_b) A.out.outlier_logits_b[v] = ll1 - logsumexp2(ll0, art);
            }
          }
        }
      } else {
      // set means: one (variant, side, feature) per thread, low threads first
      for (int idx = srow; idx < nv * 2 * E; idx += 256) {
        const int seg = (int)(((unsigned)idx * inv_e) >> 16), e = idx - seg * E;
        const int j = seg >> 1, s = seg & 1;
        const int start = (int)lds_u8((s ? m_alt_start : m_ref_start) + j), cnt = (int)lds_u8((s ? m_alt_cnt : m_ref_cnt) + j);
        const unsigned src = xch + (e * XCH_LD + start) * 4;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        for (int i = 0; i < cnt; i += 4) {
          const float x0 = lds_f32(src + i * 4), x1 = lds_f32(src + i * 4 + 4), x2 = lds_f32(src + i * 4 + 8), x3 = lds_f32(src + i * 4 + 12);
          a0 += x0;
          a1 += i + 1 < cnt ? x1 : 0.f;
          a2 += i + 2 < cnt ? x2 : 0.f;
          a3 += i + 3 < cnt ? x3 : 0.f;
        }
        float* dst = s ? A.out.alt_means_be : A.out.ref_means_be;
        if (dst) dst[(long long)lds_s32(tb_var + j * 4) * E + e] = __fdividef((a0 + a1) + (a2 + a3), (float)cnt + 1e-4f);
      }
      // log-likelihood sums: one (variant, term) per thread in groups of eight lanes, HIGH threads first (the two gathers
      // run side by side on different warps); the terms of a variant meet through shuffles
      {
        const int ridx = 255 - srow;
        const int k = ridx & 7;
        for (int base = ridx & ~31; base < nv * 8; base += 256) {
          const int j = (base + (ridx & 31)) >> 3;
          const bool term = j < nv && k < K + 2;
          float acc = 0.f;
          if (term) {
            const int as = (int)lds_u8(m_alt_start + j), ac = (int)lds_u8(m_alt_cnt + j);
            const unsigned src = xch + ((MAXE + k) * XCH_LD + as) * 4;
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
            for (int i = 0; i < ac; i += 4) {
              const float x0 = lds_f32(src + i * 4), x1 = lds_f32(src + i * 4 + 4), x2 = lds_f32(src + i * 4 + 8), x3 = lds_f32(src + i * 4 + 12);
              a0 += x0;
              a1 += i + 1 < ac ? x1 : 0.f;
              a2 += i + 2 < ac ? x2 : 0.f;
              a3 += i + 3 < ac ? x3 : 0.f;
            }
            acc = (a0 + a1) + (a2 + a3);
            if (k >= 2) acc += lds_f32(sb + HC_H + offsetof(HeadConst, logw) + (k - 2) * 4);
          }
          const bool art_term = term && k >= 2;
          float art_max = art_term ? acc : -INFINITY;
#pragma unroll
          for (int m = 1; m < 8; m <<= 1) art_max = fmaxf(art_max, __shfl_xor_sync(0xffffffffu, art_max, m));
          float sacc = art_term ? expf(acc - art_max) : 0.f;
#pragma unroll
          for (int m = 1; m < 8; m <<= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, m);
          // ridx runs against the lane number: term k of the group sits in lane (lane | 7) - k
          const int lane_k0 = (lane | 7);
          const float ll0 = __shfl_sync(0xffffffffu, acc, lane_k0), ll1 = __shfl_sync(0xffffffffu, acc, lane_k0 - 1);
          if (term) {
            const long long v = lds_s32(tb_var + j * 4);
            const float art = art_max + logf(sacc);
            if (A.out.logits_bk) A.out.logits_bk[v * (K + 2) + k] = acc;
            if (k == 0 && A.out.logits_b) A.out.logits_b[v] = 20.f * tanhf((art - ll0) / 20.f);
            if (k == 1 && A.out.outlier_logits_b) A.out.outlier_logits_b[v] = ll1 - logsumexp2(ll0, art);
          }
        }
      }
      }   // !LONG
      __syncwarp();
      if (lane == 0) mbar_arrive(sb + offsetof(Shared, meta_free) + (slot * 2 + (round & 1)) * 8);   // the tile's tables may be refilled
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc<TMEM_COLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// Tile planner: greedy packing of whole variants into tiles of <= TILE rows (ref rows padded to 4, then alt rows;
// same rule as build_tile in pmt_tile.cuh, so the set of "long" variants left to reads_forward_long_kernel is the
// same).  One warp per claim of PLAN_CLAIM consecutive variants; tiles never span claims.  tiles[0] = tile count
// (reserved with one atomicAdd per claim: tile ORDER is arbitrary, results do not depend on it).
// ------------------------------------------------------------------------------------------------
// `stage` != nullptr (training): the claim's tiles go to its own region [claim][2 * claim_variants] and their number to
// counts[claim]; compact_tiles_kernel then lists them in claim order, so the list -- and with it the order in which the
// backward sums every gradient -- is the same from run to run.
__global__ void plan_tiles_kernel(const long long* __restrict__ ref_off, const long long* __restrict__ alt_off, int B, int claim_variants,
                                  int max_nv, int* __restrict__ tiles, int* __restrict__ counts, int* __restrict__ stage) {
  __shared__ int buf[4][2 * PLAN_CLAIM];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int claim = blockIdx.x * 4 + w;
  const long long c0 = (long long)claim * claim_variants;
  if (c0 >= B) return;
  const int c1 = (int)min((long long)B, c0 + claim_variants);
  int v = (int)c0, n = 0;
  while (v < c1) {
    const long long r_base = __ldg(ref_off + v), a_base = __ldg(alt_off + v);
    int nv = 0;
    for (int base = 0; base < TILE; base += 32) {
      const int cand = v + base + lane + 1;   // tile would cover [v, cand)
      int fits = 0;
      if (cand <= c1 && base + lane < max_nv) {
        const long long nr = __ldg(ref_off + cand) - r_base, na = __ldg(alt_off + cand) - a_base;
        fits = (((nr + 3) & ~3LL) + na <= TILE) ? 1 : 0;
      }
      const unsigned ballot = __ballot_sync(0xffffffffu, fits);
      nv += __popc(ballot);
      if (ballot != 0xffffffffu) break;
    }
    if (nv == 0) { v += 1; continue; }   // longer than a tile: reads_forward_long_kernel
    if (lane == 0) { buf[w][2 * n] = v; buf[w][2 * n + 1] = nv; }
    ++n;
    v += nv;
  }
  __syncwarp();
  if (stage) {
    if (lane == 0) counts[claim] = n;
    for (int i = lane; i < 2 * n; i += 32) stage[(size_t)claim * 2 * claim_variants + i] = buf[w][i];
    return;
  }
  int base = 0;
  if (lane == 0) base = atomicAdd(tiles, n);
  base = __shfl_sync(0xffffffffu, base, 0);
  for (int i = lane; i < 2 * n; i += 32) tiles[2 + 2 * base + i] = buf[w][i];
}

// Packed planner (inference): the variants of a claim are re-ordered so that the tiles fill up -- best fit: every tile takes,
// again and again, the largest remaining set that still fits -- instead of being cut from the batch order (91.5 % -> 96 % of
// the rows of a tile used on the WGS-shaped bench data, i.e. 4.8 % fewer tiles).  A tile is then a range [p0, p0 + nv) of
// the permutation `perm` (positions are claim-local + claim base: perm[c0 + k] = k-th variant placed by claim c0).  Results
// do not depend on the composition of a tile (there is no arithmetic across the sets of a tile).  One warp per claim:
// counting sort by set size with deterministic ranks (match_any), then lane 0 places the sets with a bit mask of the
// non-empty sizes (the largest size <= space is one clz).
__global__ void __launch_bounds__(128) plan_tiles_packed_kernel(const long long* __restrict__ ref_off, const long long* __restrict__ alt_off,
                                                                int B, int claim_variants, int* __restrict__ tiles, int* __restrict__ perm) {
  __shared__ unsigned short s_order[4][PLAN_CLAIM], s_perm[4][PLAN_CLAIM];
  __shared__ unsigned short s_ra[4][PLAN_CLAIM];          // ref rows | alt rows << 8 of a claim's variant
  __shared__ int s_bucket[4][TILE + 1];                   // per set size: position of its next unused entry in s_order << 16 | entries left
  __shared__ int s_tiles[4][2 * PLAN_CLAIM];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int claim = blockIdx.x * 4 + w;
  const long long c0 = (long long)claim * claim_variants;
  if (c0 >= B) return;
  const int n = (int)min((long long)claim_variants, (long long)B - c0);
  unsigned short* order = s_order[w];
  unsigned short* ra = s_ra[w];
  int* bucket = s_bucket[w];
  int* fill = s_tiles[w];   // scratch of the counting sort (the tile list is written later)
  for (int i = lane; i <= TILE; i += 32) { bucket[i] = 0; fill[i] = 0; }
  __syncwarp();
  // sizes; a set that does not fit a tile by itself is left out (size 255: the long-set path takes it)
  int my_size[PLAN_CLAIM / 32];
#pragma unroll
  for (int k = 0; k < PLAN_CLAIM / 32; ++k) {
    const int i = k * 32 + lane;
    int size = 255;
    if (i < n) {
      const long long nr = __ldg(ref_off + c0 + i + 1) - __ldg(ref_off + c0 + i), na = __ldg(alt_off + c0 + i + 1) - __ldg(alt_off + c0 + i);
      if (((nr + 3) & ~3LL) + na <= TILE) { size = (int)(nr + na); ra[i] = (unsigned short)(nr | (na << 8)); }
    }
    my_size[k] = size;
    if (size <= TILE) atomicAdd(&bucket[size], 1);
  }
  __syncwarp();
  // bucket ranges (warp scan over the 129 sizes) and the masks of the non-empty sizes: lo = sizes 0..63, hi = 64..127
  unsigned long long lo = 0, hi = 0;
  int has128 = 0, total = 0;
  {
    int carry = 0;
    for (int s0 = 0; s0 <= TILE; s0 += 32) {
      const int sz = s0 + lane;
      const int c = sz <= TILE ? bucket[sz] : 0;
      int inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
      if (sz <= TILE) bucket[sz] = ((carry + inc - c) << 16) | c;
      const unsigned nz = __ballot_sync(0xffffffffu, c > 0);
      if (s0 == 0) lo |= nz; else if (s0 == 32) lo |= (unsigned long long)nz << 32; else if (s0 == 64) hi |= nz;
      else if (s0 == 96) hi |= (unsigned long long)nz << 32; else has128 = nz & 1;
      carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    total = carry;
  }
  __syncwarp();
  // scatter in batch order (the rank inside a bucket is the variant's rank among the variants of its size)
#pragma unroll
  for (int k = 0; k < PLAN_CLAIM / 32; ++k) {
    const int size = my_size[k];
    const unsigned peers = __match_any_sync(0xffffffffu, size);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (size <= TILE) order[(bucket[size] >> 16) + fill[size] + rank] = (unsigned short)(k * 32 + lane);
    __syncwarp();
    if (size <= TILE && rank == 0) fill[size] += __popc(peers);
    __syncwarp();
  }
  int n_tiles = 0, placed = 0;
  if (lane == 0) {
    int remaining = total;
    while (remaining > 0) {
      int nr = 0, na = 0, nv = 0;
      const int p0 = placed;
      int limit = TILE;
      while (nv < TILE) {
        // largest non-empty size <= min(limit, free rows)
        int cap = TILE - (nr + na);
        if (cap > limit) cap = limit;
        if (cap < 0) break;
        int sz = -1;
        if (cap >= TILE && has128) sz = TILE;
        else {
          const int ch = min(cap, 127) - 64;
          const unsigned long long h = ch >= 0 ? hi & (~0ull >> (63 - ch)) : 0ull;
          if (h) sz = 127 - __clzll((long long)h);
          else {
            const unsigned long long l = lo & (~0ull >> (63 - min(cap, 63)));
            if (l) sz = 63 - __clzll((long long)l);
          }
        }
        if (sz < 0) break;
        // Best fit keeps taking this size while it fits (no larger size can start to fit as the space shrinks), so up to
        // GROUP of its entries are read at once -- independent loads instead of one dependent chain per set
        constexpr int GROUP = 6;
        const int pc = bucket[sz], pos = pc >> 16, cnt = pc & 0xFFFF;
        int want = sz > 0 ? cap / sz : GROUP;
        if (want > cnt) want = cnt;
        if (want > TILE - nv) want = TILE - nv;
        if (want > GROUP) want = GROUP;
        int ids[GROUP], rvs[GROUP];
#pragma unroll
        for (int j = 0; j < GROUP; ++j) ids[j] = j < want ? order[pos + j] : 0;
#pragma unroll
        for (int j = 0; j < GROUP; ++j) rvs[j] = j < want ? ra[ids[j]] : 0;
        int took = 0;
#pragma unroll
        for (int j = 0; j < GROUP; ++j) {
          if (j < want && took == j) {
            const int r = rvs[j] & 255, a = rvs[j] >> 8;
            if (((nr + r + 3) & ~3) + na + a <= TILE) {
              s_perm[w][placed + j] = (unsigned short)ids[j];
              nr += r; na += a; took = j + 1;
            }
          }
        }
        if (took > 0) {
          placed += took; nv += took; remaining -= took;
          bucket[sz] = pc + took * 65535;   // position + took, entries left - took
          if (cnt == took) {                // the size is used up
            if (sz == TILE) has128 = 0;
            else if (sz >= 64) hi &= ~(1ull << (sz - 64));
            else lo &= ~(1ull << sz);
          }
          limit = took == want ? TILE : sz - 1;   // stopped early: the next one of this size did not fit (padding) -> smaller sizes
        } else {
          limit = sz - 1;   // the padding of the ref rows made it too long: try the next smaller size
        }
      }
      s_tiles[w][2 * n_tiles] = (int)c0 + p0; s_tiles[w][2 * n_tiles + 1] = nv;
      ++n_tiles;
    }
  }
  n_tiles = __shfl_sync(0xffffffffu, n_tiles, 0);
  placed = __shfl_sync(0xffffffffu, placed, 0);
  int base = 0;
  if (lane == 0) base = atomicAdd(tiles, n_tiles);
  base = __shfl_sync(0xffffffffu, base, 0);
  for (int i = lane; i < 2 * n_tiles; i += 32) tiles[2 + 2 * base + i] = s_tiles[w][i];
  for (int i = lane; i < placed; i += 32) perm[c0 + i] = (int)c0 + s_perm[w][i];
}

// One CTA: exclusive scan of the per-claim tile counts, then the claims' tiles copied behind each other.
__global__ void compact_tiles_kernel(const int* __restrict__ counts, const int* __restrict__ stage, int n_claims, int claim_variants,
                                     int* __restrict__ tiles) {
  __shared__ int warp_tot[32];
  __shared__ int running;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0) running = 0;
  __syncthreads();
  for (int c0 = 0; c0 < n_claims; c0 += blockDim.x) {
    const int c = c0 + tid;
    const int n = c < n_claims ? counts[c] : 0;
    int inc = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) warp_tot[w] = inc;
    __syncthreads();
    int before = running;
    for (int i = 0; i < w; ++i) before += warp_tot[i];
    const int first = before + inc - n;
    for (int i = 0; i < 2 * n; ++i) tiles[2 + 2 * first + i] = stage[(size_t)c * 2 * claim_variants + i];
    __syncthreads();
    if (tid == blockDim.x - 1) running = before + inc;
    __syncthreads();
  }
  if (tid == 0) tiles[0] = running;
}

// ------------------------------------------------------------------------------------------------
// Long-set tile list (pmt_tc.cuh: LongTile).  long_list_kernel appends every set plan_tiles_kernel leaves out (same rule:
// pad4(ref rows) + alt rows > TILE) to a list, in arbitrary order; long_layout_kernel places the sets' tiles so that no
// set straddles a round of R slots (padding tiles fill the gaps: the array is preset to -1) and writes the descriptors.
// ------------------------------------------------------------------------------------------------
__global__ void long_list_kernel(const long long* __restrict__ ref_off, const long long* __restrict__ alt_off, int B, int cap,
                                 int* __restrict__ list) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < B; v += gridDim.x * blockDim.x) {
    const long long nr = __ldg(ref_off + v + 1) - __ldg(ref_off + v), na = __ldg(alt_off + v + 1) - __ldg(alt_off + v);
    if (((nr + 3) & ~3LL) + na > TILE) {
      const int i = atomicAdd(list, 1);
      if (i < cap) list[1 + i] = v;
    }
  }
}

__global__ void long_layout_kernel(const long long* __restrict__ ref_off, const long long* __restrict__ alt_off, const int* __restrict__ list,
                                   int cap, int R, int max_tiles, LongTile* __restrict__ tiles, int* __restrict__ n_tiles) {
  __shared__ __align__(16) int s_T[1024], s_first[1024];
  __shared__ int s_pos;
  const int tid = threadIdx.x;
  const int n = min(list[0], cap);
  if (tid == 0) s_pos = 0;
  __syncthreads();
  for (int c0 = 0; c0 < n; c0 += blockDim.x) {
    const int i = c0 + tid;
    int v = -1, nr = 0, na = 0, tr = 0, ta = 0;
    if (i < n) {
      v = list[1 + i];
      nr = (int)(__ldg(ref_off + v + 1) - __ldg(ref_off + v)); na = (int)(__ldg(alt_off + v + 1) - __ldg(alt_off + v));
      tr = (nr + TILE - 1) / TILE; ta = (na + TILE - 1) / TILE;
    }
    s_T[tid] = tr + ta;
    __syncthreads();
    if (tid == 0) {
      // the only sequential part: positions with round padding (running `room` = slots left in the round, no divisions)
      int pos = s_pos, room = R - pos % R;
      const int m = min((int)blockDim.x, n - c0);
      for (int j0 = 0; j0 < m; j0 += 4) {
        const int4 t4 = *reinterpret_cast<const int4*>(s_T + j0);
        const int tt[4] = {t4.x, t4.y, t4.z, t4.w};
        int f[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int T = tt[q];
          if (j0 + q >= m || T > R) { f[q] = -1; continue; }   // T > R: host-side guard, never taken
          if (T > room) { pos += room; room = R; }
          f[q] = pos;
          pos += T; room -= T;
          if (room == 0) room = R;
        }
        *reinterpret_cast<int4*>(s_first + j0) = make_int4(f[0], f[1], f[2], f[3]);
      }
      s_pos = pos;
    }
    __syncthreads();
    if (i < n) {
      const int first = s_first[tid];
      if (first >= 0 && first + tr + ta <= max_tiles) {
        for (int k = 0; k < tr + ta; ++k) {
          const int side = k < tr ? 0 : 1, kk = side ? k - tr : k;
          LongTile t;
          t.v = v; t.side = side; t.start = kk * TILE; t.cnt = min(TILE, (side ? na : nr) - kk * TILE);
          t.k = k; t.first = first; t.t_ref = tr; t.t_alt = ta;
          tiles[first + k] = t;
        }
      }
    }
    __syncthreads();
  }
  if (tid == 0) *n_tiles = min(s_pos, max_tiles);
}

// ------------------------------------------------------------------------------------------------
// Weight images: for every step the logical B matrix [N][K] (N = output column of the MMA, K = operand column),
// K-major with the 128-byte swizzle, K blocks of 32 elements; hi = TF32-rounded value, lo = remainder.
// ------------------------------------------------------------------------------------------------
__global__ void pack_tc_kernel(const __grid_constant__ PmtModelDesc D, const __grid_constant__ TcPlan TP, const float* __restrict__ w,
                               unsigned char* __restrict__ image) {
  const TcStep& o = TP.step[blockIdx.x];
  const int K = o.KS * 8;
  const int n_kb = (K + 31) / 32;
  for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < n_kb * o.N * 32; idx += gridDim.y * blockDim.x) {
    const int kb = idx / (o.N * 32), rem = idx % (o.N * 32), n = rem / 32, kk = rem % 32;
    const int k = kb * 32 + kk;
    const float v = k < K ? tc_weight(D, o, w, n, k) : 0.f;
    const float hi = rna_tf32(v);
    const float lo = v - hi;
    const unsigned L = (unsigned)n * 128u + (unsigned)kk * 4u;
    const unsigned phys = L ^ (((L >> 7) & 7u) << 4);
    const size_t off = (size_t)o.img_off + (size_t)kb * o.N * 128 + phys;
    *reinterpret_cast<float*>(image + off) = hi;
    *reinterpret_cast<float*>(image + off + o.img_bytes) = lo;
  }
}

}  // namespace tc
}  // namespace pmt

// ================================================================================================
// host side
// ================================================================================================
using namespace pmt;
using namespace pmt::tc;

static int g_precision = PMT_PRECISION_FP32;
extern "C" int pmt_set_precision(int mode) {
  PMT_CHECK(mode == PMT_PRECISION_FP32 || mode == PMT_PRECISION_TF32X3 || mode == PMT_PRECISION_TF32,
            "unknown precision mode %d", mode);
  g_precision = mode;
  return 0;
}
extern "C" int pmt_get_precision(void) { return g_precision; }
int pmt_precision_mode() { return g_precision; }

static int pad_to(int v, int m) { return (v + m - 1) / m * m; }

// Shape envelope of the tensor-core kernel.  Read program: Linear+SELU then DenseSkipBlocks of width d_read <= 31;
// reducer: DenseSkipBlocks of width d_model then one Linear to d_feat; d_model = d_read + d_info + d_seq with
// d_info + d_seq <= 32 (column 31 of every 64-wide operand carries the bias).
bool pmt_tc_supported(const Plan& P) {
  const PmtModelDesc& d = P.d;
  if (d.n_read_features > 61 || d.read_row_bytes > 12 || d.d_read > 31 || d.d_info + d.d_seq > 32 ||
      d.d_model != d.d_read + d.d_info + d.d_seq || d.d_ffn / 2 > MAXH || d.d_ffn % 2 || d.d_feat > MAXE || d.n_clusters > MAXK ||
      d.n_blocks < 1)
    return false;
  if (d.n_read_ops < 2 || !(d.read_ops[0].flags & PMT_OP_POST_SELU) || (d.read_ops[0].flags & (PMT_OP_SKIP_BEGIN | PMT_OP_SKIP_END)) ||
      d.read_ops[0].in_dim != d.n_read_features || d.read_ops[0].out_dim != d.d_read)
    return false;
  bool inside = false;
  for (int i = 1; i < d.n_read_ops; ++i) {
    const PmtLinearOp& o = d.read_ops[i];
    if (o.in_dim != d.d_read || o.out_dim != d.d_read) return false;
    if (!inside && !(o.flags & PMT_OP_SKIP_BEGIN)) return false;
    inside = !(o.flags & PMT_OP_SKIP_END);
  }
  if (inside) return false;
  if (d.n_red_ops < 1) return false;
  for (int i = 0; i + 1 < d.n_red_ops; ++i) {
    const PmtLinearOp& o = d.red_ops[i];
    if (o.in_dim != d.d_model || o.out_dim != d.d_model) return false;
    if (!inside && !(o.flags & PMT_OP_SKIP_BEGIN)) return false;
    inside = !(o.flags & PMT_OP_SKIP_END);
  }
  if (inside) return false;
  const PmtLinearOp& last = d.red_ops[d.n_red_ops - 1];
  if (last.flags != 0 || last.in_dim != d.d_model || last.out_dim != d.d_feat) return false;
  return d.n_read_ops + 2 * d.n_blocks + d.n_red_ops <= MAX_STEPS;
}

static TcStep& add_step(TcPlan& T, int epi, int N, int K, int dst_x) {
  TcStep& o = T.step[T.n_steps++];
  memset(&o, 0, sizeof(o));
  o.epi = epi; o.N = N; o.KS = K / 8; o.dst_x = dst_x;
  o.alpha_off = -1; o.bias_col = -1;
  T.image_bytes = pad_to(T.image_bytes, 1024);
  o.img_off = T.image_bytes;
  o.img_bytes = ((K + 31) / 32) * N * 128;
  T.image_bytes += 2 * o.img_bytes;
  if (2 * o.img_bytes > T.slot_bytes) T.slot_bytes = 2 * o.img_bytes;
  return o;
}

static void linear_step(TcStep& o, const PmtLinearOp& l, int k_perm, int n_perm, int k_selu_scale, int bias_col) {
  o.pk = PK_LINEAR; o.k_real = l.in_dim; o.n_real = l.out_dim; o.w_off = l.w_off; o.b_off = l.b_off;
  o.alpha_off = (l.flags & PMT_OP_SKIP_END) ? l.alpha_off : -1;
  o.k_perm = k_perm; o.n_perm = n_perm; o.k_selu_scale = k_selu_scale; o.bias_col = bias_col;
}

void pmt_tc_plan(const Plan& P, TcPlan* out) {
  TcPlan& T = *out;
  memset(&T, 0, sizeof(T));
  const PmtModelDesc& d = P.d;
  const int H = d.d_ffn / 2;
  // read embedding (mlp.py:25-76)
  linear_step(add_step(T, EPI_DECODE, 32, 64, 0), d.read_ops[0], 0, 0, 0, 63);
  for (int i = 1; i < d.n_read_ops; ++i) {
    const PmtLinearOp& l = d.read_ops[i];
    const int epi = (l.flags & PMT_OP_SKIP_BEGIN) ? (i == 1 ? EPI_FIRST32 : EPI_ACT_X32) : EPI_ACT_Z32;
    linear_step(add_step(T, epi, 32, 32, (l.flags & PMT_OP_SKIP_END) ? 1 : 0), l, 0, 0, 1, 31);
  }
  // gated blocks (gated_mlp.py:177-251)
  for (int b = 0; b < d.n_blocks; ++b) {
    TcStep& p1 = add_step(T, b == 0 ? EPI_LN_FIRST : EPI_LN, 2 * NP1, 64, 0);
    p1.pk = PK_PROJ1; p1.blk = b; p1.bias_col = 31;
    TcStep& p2 = add_step(T, EPI_GATE, 64, 24, 1);
    p2.pk = PK_PROJ2; p2.blk = b;
    (void)H;
  }
  // reducer (artifact_model.py:258-259) + rotation (euclidean_transformation.py:19-20)
  for (int i = 0; i + 1 < d.n_red_ops; ++i) {
    const PmtLinearOp& l = d.red_ops[i];
    const int epi = (l.flags & PMT_OP_SKIP_BEGIN) ? EPI_ACT_X64 : EPI_ACT_Z64;
    linear_step(add_step(T, epi, 64, 64, (l.flags & PMT_OP_SKIP_END) ? 1 : 0), l, 1, 1, 1, 31);
  }
  {
    const PmtLinearOp& l = d.red_ops[d.n_red_ops - 1];
    TcStep& o = add_step(T, EPI_COPY_X64, 16, 64, 0);
    o.pk = PK_FINAL; o.k_real = l.in_dim; o.n_real = l.out_dim; o.w_off = l.w_off; o.b_off = l.b_off; o.bias_col = 31;
  }
  T.image_bytes = pad_to(T.image_bytes, 1024);

  // ---- training: saved operands, backward program, gradient accumulators (pmt_tc_bwd.cu) ----
  int scr = 0, timg = 0, part = 0;
  for (int s = 0; s < T.n_steps; ++s) {
    TcStep& o = T.step[s];
    const int width = o.KS * 8, n_panels = (width + 31) / 32;
    o.scr_off = scr; o.scr_bytes = n_panels * PANEL_BYTES; scr += o.scr_bytes;
    o.Nd = pad_to(width, 16); o.KSd = o.N / 8;
    o.t_img_off = timg;
    o.t_img_bytes = s == 0 ? 0 : ((o.N + 31) / 32) * o.Nd * 128;   // the first layer's input is data: no data gradient
    timg += pad_to(o.t_img_bytes, 1024);
    if (o.t_img_bytes > T.t_stage_bytes) T.t_stage_bytes = o.t_img_bytes;
    o.kw = 32 * n_panels; o.part_off = part; part += o.N * o.kw;
    if (s + 1 == T.n_steps) { o.bepi = BE_HEAD; continue; }
    switch (T.step[s + 1].epi) {
      case EPI_COPY_X64: o.bepi = BE_GINIT64; break;
      case EPI_ACT_Z64: o.bepi = BE_DZ64; break;
      case EPI_ACT_X64: o.bepi = BE_GACC64; break;
      case EPI_GATE: o.bepi = BE_GATE; break;
      case EPI_LN: o.bepi = BE_LN64; break;
      case EPI_LN_FIRST: o.bepi = BE_LN_EMBED; break;
      case EPI_ACT_Z32: o.bepi = BE_DZ32; break;
      case EPI_ACT_X32: o.bepi = BE_GACC32; break;
      default: o.bepi = BE_FIRST; break;   // EPI_FIRST32
    }
  }
  T.t_image_bytes = pad_to(timg, 1024);
  T.x0_off = scr; scr += 32 * TILE * (int)sizeof(float);
  T.f_off = scr; scr += MAXE * TILE * (int)sizeof(float);
  T.rstd_off = scr; scr += d.n_blocks * TILE * (int)sizeof(float);
  T.gate_off = scr; scr += d.n_blocks * GATE_ITEMS * 2 * TILE * (int)sizeof(float);
  T.means_off = scr; scr += d.n_blocks * 2 * BWD_MAXV * MAXH * (int)sizeof(float);
  T.tile_bytes = pad_to(scr, 1024);
  T.scal_off = part;
  T.part_floats = pad_to(part + 8 * SCAL_W, 64);
}

int pmt_plan_claim_variants(int n_variants, int n_sm) {
  // planner claims: large enough that the partial last tile of a claim is a small loss, small enough that a small
  // batch is planned by many warps (each claim is walked sequentially)
  int claim_variants = n_variants / (2 * n_sm);
  if (claim_variants < 64) claim_variants = 64;
  if (claim_variants > PLAN_CLAIM) claim_variants = PLAN_CLAIM;
  return claim_variants;
}
size_t pmt_plan_claim_bytes(int n_variants, int n_sm) {
  const int cv = pmt_plan_claim_variants(n_variants, n_sm);
  const size_t n_claims = ((size_t)n_variants + cv - 1) / cv;
  return (n_claims * (1 + 2 * (size_t)cv) * sizeof(int) + 255) & ~(size_t)255;
}
// Tile list of a batch: tiles[0] = count, (first variant, variants) pairs from tiles[2].  deterministic: the list order is
// fixed (claim order); claim_buf: pmt_plan_claim_bytes() bytes.
int pmt_plan_tiles(const PmtBatch* batch, int max_variants, bool deterministic, int n_sm, int* tiles, int* claim_buf, int* n_claims_out,
                   cudaStream_t st) {
  const int claim_variants = pmt_plan_claim_variants(batch->n_variants, n_sm);
  const int n_claims = (batch->n_variants + claim_variants - 1) / claim_variants;
  if (n_claims_out) *n_claims_out = n_claims;
  const long long* ro = reinterpret_cast<const long long*>(batch->ref_off);
  const long long* ao = reinterpret_cast<const long long*>(batch->alt_off);
  if (!deterministic) {
    PMT_CUDA(cudaMemsetAsync(tiles, 0, 2 * sizeof(int), st));
    plan_tiles_kernel<<<(n_claims + 3) / 4, 128, 0, st>>>(ro, ao, batch->n_variants, claim_variants, max_variants, tiles, nullptr, nullptr);
    return 0;
  }
  int* counts = claim_buf;
  int* stage = claim_buf + n_claims;
  plan_tiles_kernel<<<(n_claims + 3) / 4, 128, 0, st>>>(ro, ao, batch->n_variants, claim_variants, max_variants, tiles, counts, stage);
  compact_tiles_kernel<<<1, 1024, 0, st>>>(counts, stage, n_claims, claim_variants, tiles);
  return 0;
}

// The read kernel's weight ring: as many stages as fit next to the fixed carve, at most NS_MAX.
Ring pmt_tc_ring(const TcPlan& T, int passes) {
  Ring R;
  R.stage_bytes = passes == 3 ? T.slot_bytes : T.slot_bytes / 2;
  R.n_stages = (int)((227 * 1024 - FWD_FIXED_BYTES) / R.stage_bytes);
  if (R.n_stages > NS_MAX) R.n_stages = NS_MAX;
  R.smem = FWD_FIXED_BYTES + (size_t)R.n_stages * R.stage_bytes;
  return R;
}

template <int PASSES, bool SAVE, bool LONG>
static int launch_reads_tc(const PmtModelDesc& D, const TcPlan& T, const TcArgs& A, int grid, const Ring& R, cudaStream_t st) {
  PMT_CUDA(cudaFuncSetAttribute(reads_forward_tc_kernel<PASSES, SAVE, LONG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R.smem));
  reads_forward_tc_kernel<PASSES, SAVE, LONG><<<grid, FWD_THREADS, R.smem, st>>>(D, T, A, R.n_stages, R.stage_bytes);
  return 0;
}

int pmt_launch_pack_tc(const Plan& P, const TcPlan& T, const float* weights, unsigned char* image, cudaStream_t st) {
  pack_tc_kernel<<<dim3(T.n_steps, 8), 256, 0, st>>>(P.d, T, weights, image);
  return 0;
}

// Training recompute: the forward over tiles [tile_first, tile_limit) of a planned tile list, operands saved to `scratch`
// (always the split-precision mode: the saved activations are the fp32-parity ones).
int pmt_launch_reads_tc_save(const CallPlan& C, const TcArgs& A, int grid, cudaStream_t st) {
  return launch_reads_tc<3, true, false>(C.P.d, C.T, A, grid, C.ring_save, st);
}

// Launches the tile planner, the weight packer (unless the images in W.tc_image are still valid) and the tensor-core
// read kernel.
int pmt_launch_reads_tc(const CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                        const FwdBuffers& W, bool reuse_images, cudaStream_t st) {
  const TcPlan& T = C.T;
  unsigned char* image = W.tc_image;
  int* tiles = W.tiles;
  int* perm = W.perm;
  int n_claims = 0;
  if (C.packed_planner) {
    n_claims = (batch->n_variants + PLAN_CLAIM - 1) / PLAN_CLAIM;
    PMT_CUDA(cudaMemsetAsync(tiles, 0, 2 * sizeof(int), st));
    plan_tiles_packed_kernel<<<(n_claims + 3) / 4, 128, 0, st>>>(reinterpret_cast<const long long*>(batch->ref_off),
                                                                reinterpret_cast<const long long*>(batch->alt_off), batch->n_variants,
                                                                PLAN_CLAIM, tiles, perm);
  } else if (pmt_plan_tiles(batch, TILE, false, C.n_sm, tiles, nullptr, &n_claims, st)) {
    return 1;
  }
  if (!reuse_images) pack_tc_kernel<<<dim3(T.n_steps, 8), 256, 0, st>>>(C.P.d, T, weights, image);
  TcArgs A;
  A.wflat = weights; A.image = image; A.tiles = tiles; A.perm = perm; A.batch = *batch; A.out = *out;
  A.scratch = nullptr; A.tile_first = 0; A.tile_limit = 0x7fffffff;
  // the second slot of each CTA takes a second tile once every SM has one
  const int grid = pmt_tile_grid(batch, n_claims, C.n_sm);
  pmt_profile_begin(st);
  const int rc = C.passes == 1 ? launch_reads_tc<1, false, false>(C.P.d, T, A, grid, C.ring, st)
                               : launch_reads_tc<3, false, false>(C.P.d, T, A, grid, C.ring, st);
  pmt_profile_end(st);
  return rc;
}

// ---- sets longer than a tile (pmt_tc.cuh: LongTile) ----
// The sets plan_tiles_kernel left out, on the same tensor-core pipeline (the weight images in W.tc_image must be packed:
// call after pmt_launch_reads_tc).  Every CTA of the grid has to be resident (a tile waits for the other tiles of its
// set): one CTA per SM, grid = number of SMs.
int pmt_launch_reads_tc_long(const CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                             const FwdBuffers& W, cudaStream_t st) {
  const LongLayout& L = C.long_tc;
  const LongBuffers& LB = W.lng;
  const long long* ro = reinterpret_cast<const long long*>(batch->ref_off);
  const long long* ao = reinterpret_cast<const long long*>(batch->alt_off);
  PMT_CUDA(cudaMemsetAsync(LB.list, 0, sizeof(int), st));
  PMT_CUDA(cudaMemsetAsync(LB.tiles, 0xFF, (size_t)L.max_tiles * sizeof(LongTile), st));
  PMT_CUDA(cudaMemsetAsync(LB.counters, 0, L.counters.bytes, st));
  int blocks = (batch->n_variants + 255) / 256;
  if (blocks > 4 * C.n_sm) blocks = 4 * C.n_sm;
  long_list_kernel<<<blocks, 256, 0, st>>>(ro, ao, batch->n_variants, L.cap, LB.list);
  long_layout_kernel<<<1, 1024, 0, st>>>(ro, ao, LB.list, L.cap, L.R, L.max_tiles, LB.tiles, LB.n_tiles);
  TcArgs A;
  memset(&A, 0, sizeof(A));
  A.wflat = weights; A.image = W.tc_image; A.tiles = nullptr; A.batch = *batch; A.out = *out;
  A.scratch = nullptr; A.tile_first = 0; A.tile_limit = 0x7fffffff;
  A.lng.tiles = LB.tiles; A.lng.n_tiles = LB.n_tiles;
  A.lng.mf_cnt = LB.counters;
  A.lng.fin_cnt = LB.fin_cnt;
  A.lng.mf_part = LB.mf_part;
  A.lng.fin_part = LB.fin_part;
  const int grid = L.R / 2;
  return C.passes == 1 ? launch_reads_tc<1, false, true>(C.P.d, C.T, A, grid, C.ring, st)
                       : launch_reads_tc<3, false, true>(C.P.d, C.T, A, grid, C.ring, st);
}
