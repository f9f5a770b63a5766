// Declarations shared by the tensor-core read-path kernels: the forward (pmt_tc.cu) and the backward (pmt_tc_bwd.cu).
#pragma once
#include <cstddef>
#include <cstring>

#include "pmt_host.h"
#include "pmt_tile.cuh"
#include "pmt_tc_ptx.cuh"

namespace pmt {
namespace tc {

constexpr int THREADS = 608;      // 16 epilogue warps (2 slots x 2 column halves x 4 lane quarters) + 2 MMA warps + loader warp
constexpr int MMA_WARP = 16, LOAD_WARP = 18;
constexpr int META_WARP = 19, FWD_THREADS = 640;   // forward only: one more warp prepares the NEXT tile's tables and rows
constexpr int SUMS_FLOATS = 2 * TILE * 11;   // per slot: [segment][MAXH]
constexpr int MAX_STEPS = 64;
constexpr int COL_X = 0, COL_Z = 64, COL_AHI = 128, COL_ALO = 192, SLOT_COLS = 256;
constexpr int TMEM_COLS = 2 * SLOT_COLS;   // TMEM columns of the forward and the backward CTA: both slots
constexpr int MAXH = 11;    // d_ffn / 2: the proj2 operand [t_ref | t_alt | is_ref, is_alt] must fit 24 columns
constexpr int NP1 = 24;     // padded width of one proj1 weight set (>= 2 * MAXH)
constexpr int MAXE = 16;    // final feature dimension
constexpr int MAXK = 6;     // artifact clusters
constexpr int XCH_ROWS = MAXE + MAXK + 2;
constexpr int XCH_LD = TILE + 1;   // odd row stride: the per-variant gathers read one column range of MANY rows at once
constexpr int NS_MAX = 8;
constexpr int PLAN_CLAIM = 512;   // variants per planner claim

enum EpiKind { EPI_DECODE = 0, EPI_FIRST32, EPI_ACT_Z32, EPI_ACT_X32, EPI_LN_FIRST, EPI_LN, EPI_GATE, EPI_ACT_X64,
               EPI_ACT_Z64, EPI_COPY_X64 };
enum PackKind { PK_LINEAR = 0, PK_PROJ1, PK_PROJ2, PK_FINAL };
// Backward epilogue that turns the data gradient coming out of step s + 1 into dL/d(output of step s) (pmt_tc_bwd.cu)
enum BwdEpi { BE_HEAD = 0, BE_GINIT64, BE_DZ64, BE_GACC64, BE_GATE, BE_LN64, BE_LN_EMBED, BE_DZ32, BE_GACC32, BE_FIRST };

// ---- training recompute: what the forward leaves in global memory for the tensor-core backward ----
// An operand of W features is saved as ceil(W / 32) PANELS of [TILE rows][32 floats] (128 bytes per row) whose 32-byte
// units are XOR-swizzled with row % 4: tcgen05's SWIZZLE_128B_BASE32B layout, the only one an MN-major tf32 operand may
// have (profiles/microbench/wgrad_probe.cu).  A panel is copied to shared memory with one bulk copy and is then the A
// operand of the weight-gradient MMA (reduction over the tile's rows) as it lies.
constexpr int PANEL_BYTES = TILE * 128;
constexpr int GATE_ITEMS = 19;     // per (row, half) of a gated block: z1[6], xhat2[6], selu'(z2)[6], rstd2
constexpr int BWD_MAXV = 32;       // variants per tile when the tile list is planned for training
constexpr int SCAL_BLOCK = 24;     // per-warp scalar gradient slots of one gated block
constexpr int SCAL_HEAD = 16 + 128;
constexpr int SCAL_W = PMT_MAX_BLOCKS * SCAL_BLOCK + SCAL_HEAD;
__host__ __device__ __forceinline__ unsigned panel_off(int row, int chunk) {   // byte offset of 16-byte chunk `chunk` of `row`
  return (unsigned)((chunk >> 3) * PANEL_BYTES + row * 128 + ((((chunk & 7) >> 1) ^ (row & 3)) << 5) + (chunk & 1) * 16);
}

struct TcStep {
  int epi;          // epilogue kind that PRODUCES this step's A operand
  int N, KS;        // MMA shape: N columns (multiple of 8), KS k-steps of 8
  int dst_x;        // 1: accumulate into X, 0: overwrite Z
  int img_off;      // byte offset of the hi image (1024-aligned); the lo image follows at + img_bytes
  int img_bytes;    // bytes of ONE image
  int blk;          // gated block of EPI_LN* / EPI_GATE
  // packing
  int pk, k_real, n_real, w_off, b_off, alpha_off, k_perm, n_perm, k_selu_scale, bias_col;
  // training: saved operand (byte offset / bytes inside a tile's scratch), backward program
  int scr_off, scr_bytes;
  int bepi;         // BwdEpi producing dL/d(output of this step)
  int Nd, KSd;      // data-gradient MMA: N = operand width padded to 16, k-steps = N / 8
  int t_img_off, t_img_bytes;   // transposed image (hi part only) inside the backward image buffer
  int part_off, kw; // weight-gradient accumulator [N][kw] (floats) inside a slot's private gradient buffer
};

struct TcPlan {
  int n_steps;
  int image_bytes;   // total bytes of the image buffer
  int slot_bytes;    // bytes of one ring stage for the x3 mode (largest hi + lo image)
  // training scratch of one tile (bytes): operand panels (TcStep.scr_off), then
  int x0_off;        // [32][TILE]  read embedding before the first DenseSkipBlock
  int f_off;         // [MAXE][TILE] final features
  int rstd_off;      // [n_blocks][TILE] LayerNorm 1/std of each gated block
  int gate_off;      // [n_blocks][GATE_ITEMS][2][TILE]
  int means_off;     // [n_blocks][2 * BWD_MAXV][MAXH] mean fields
  int tile_bytes;
  int t_image_bytes, t_stage_bytes;   // backward images: total, largest
  int part_floats;   // floats of one slot's private gradient buffer: step accumulators, then [8 warps][SCAL_W] scalars
  int scal_off;
  TcStep step[MAX_STEPS];
};

// ---- sets longer than a tile on the tensor-core forward (reads_forward_tc_kernel<.., LONG = true>) ----
// A long set is cut into tiles of <= TILE rows of ONE side (all its ref tiles, then all its alt tiles, at consecutive
// positions [first, first + t_ref + t_alt) of the long-tile list).  The tiles of a set are in flight at the same time -- the
// list is padded so that a set never straddles a round of 2 x grid slots -- and meet twice per gated block and once at
// the end through global memory: every tile leaves its partial column sums in its own slot, bumps the set's counter, waits
// for the counter to reach the set's tile count and adds the partials up in tile order (bitwise reproducible).  That is the
// whole cross-read coupling of the model (gated_mlp.py:236-248, ragged_sets.py:144-158).
struct LongTile {
  int v;        // variant (-1: padding tile)
  int side;     // 0 = ref rows, 1 = alt rows
  int start;    // first row of the tile inside the set's side
  int cnt;      // rows
  int k;        // index of the tile inside its set (ref tiles first)
  int first;    // position of the set's first tile in the list
  int t_ref, t_alt;
};
constexpr int LONG_FIN_W = MAXE + MAXK + 2;   // per tile: feature sums, then the K + 2 log-likelihood sums (alt tiles)
struct LongArgs {
  const LongTile* tiles;
  const int* n_tiles;      // device: list length incl. padding tiles
  float* mf_part;          // [tile][n_blocks][MAXH] column sums of the normalised z2 of the tile's rows
  int* mf_cnt;             // [first][n_blocks] arrival counters (zeroed before the launch)
  float* fin_part;         // [tile][LONG_FIN_W]
  int* fin_cnt;            // [first]
};

struct TcArgs {
  const float* wflat;
  const unsigned char* image;
  const int* tiles;       // [0] = number of tiles, then (v0, nv) pairs from entry 2
  const int* perm;        // packed planner: a tile covers positions [v0, v0 + nv) of this variant list; NULL: variants [v0, v0 + nv)
  PmtBatch batch;
  PmtOutputs out;
  // training recompute (SAVE kernels): tiles [tile_first, tile_limit) of the list, scratch of tile t at
  // scratch + (t - tile_first) * TcPlan.tile_bytes
  unsigned char* scratch;
  int tile_first, tile_limit;
  LongArgs lng;           // LONG kernels only
};

struct TcBwdArgs {
  const float* wflat;
  const unsigned char* image_t;   // transposed weight images
  const int* tiles;
  PmtBatch batch;
  const float* d_logits_bk;       // upstream gradients (may be null)
  const float* d_alt_means;
  const float* d_ref_means;
  float* d_info_seq;              // [B][d_info + d_seq]
  const unsigned char* scratch;
  int tile_first, tile_limit;
  float* partials;                // [2 * grid][TcPlan.part_floats]: slot s of CTA b owns buffer 2 b + s
};

struct SlotMeta {
  unsigned char rowvar[TILE];   // local variant of each row, 255 = padding
  unsigned char ref_start[TILE], ref_cnt[TILE], alt_start[TILE], alt_cnt[TILE];
};

// What the forward's meta warp prepares for a tile while the previous tile of the slot is still being computed
struct TileBuf {
  long long idx[TILE];         // batch row of each tile row (-1: padding)
  long long src[TILE];         // row of the reads array (idx through the gather indices of a downsampled / dataset-order batch)
  unsigned words[TILE * 3];    // the compressed row itself (12-byte rows)
  int var[TILE];               // the tile's variants (tile list position -> variant through the planner's permutation)
  int v0, nv, ref_pad, pad_;
  int lt[8];                   // LONG: first, k, t_ref, t_alt, side, rows, set's ref reads, set's alt reads
  SlotMeta m;
};

struct Shared {
  unsigned long long bar_a[2], bar_d[2], wfull[NS_MAX], wfree[NS_MAX];
  unsigned long long meta_full[2][2], meta_free[2][2];   // [slot][buffer]
  unsigned tmem_base;
  int pad_;
  TileBuf tb[2][2];  // [slot][round & 1]
};

// Forward head constants in shared memory: the clustering head's (pmt_tile.cuh) plus reciprocals and the cluster directions
struct HeadConstTc {
  HeadConst h;
  float inv_sigma[MAXE];
  float unit[MAXK][MAXE];
  float inv_two_tau2[MAXK], inv_sqrt2_sigma[MAXK];
};

// per gated block scalars staged in shared memory (gated_mlp.py:213-226)
constexpr int BC_LN2W = 0, BC_LN2B = 12, BC_REG = 24, BC_AREF = 36, BC_AALT = 37, BC_BREF = 38, BC_BALT = 39, BC_GAMMA = 40,
              BC_REGW = 41, BC_STRIDE = 48;

// Dynamic shared memory of the forward: the regions below at fixed byte offsets from one 8-aligned base, then the weight
// ring (the only runtime-sized region) at FWD_RING, 1024-aligned.  Every epilogue address is the base plus a constant.
constexpr unsigned FWD_XCH = (sizeof(Shared) + 7) & ~7u;                            // [2 slots][XCH_ROWS][XCH_LD] floats
constexpr unsigned FWD_SUMS = FWD_XCH + 2 * XCH_ROWS * XCH_LD * 4;                  // [2 slots][SUMS_FLOATS]
constexpr unsigned FWD_PAIRX = FWD_SUMS + 2 * SUMS_FLOATS * 4;                      // [2 slots][2 halves][TILE] float2
constexpr unsigned FWD_BLKC = FWD_PAIRX + 2 * 2 * TILE * 2 * 4;                     // [PMT_MAX_BLOCKS][BC_STRIDE] floats
constexpr unsigned FWD_HEAD = FWD_BLKC + PMT_MAX_BLOCKS * BC_STRIDE * 4;            // HeadConstTc
constexpr unsigned FWD_STEPS = FWD_HEAD + sizeof(HeadConstTc);                      // [MAX_STEPS] bytes: epi | blk << 4
constexpr unsigned FWD_RING = (FWD_STEPS + MAX_STEPS + 7) & ~7u;
// what the launch reserves next to the ring (the base is found by rounding the ring's start up to 1024)
constexpr size_t FWD_FIXED_BYTES = 2 * XCH_ROWS * XCH_LD * sizeof(float) + 2 * SUMS_FLOATS * sizeof(float) + 2 * 2 * TILE * 2 * sizeof(float) +
                                   PMT_MAX_BLOCKS * BC_STRIDE * sizeof(float) + sizeof(HeadConstTc) + sizeof(Shared) + 1024 + 64;
static_assert(FWD_RING + 1023 <= FWD_FIXED_BYTES, "forward shared-memory carve exceeds the launch's reservation");
static_assert(EPI_COPY_X64 < 16 && PMT_MAX_BLOCKS <= 16, "step table packs epi and blk into 4 bits each");

template <int NC>
__device__ __forceinline__ void tmem_st_n(unsigned taddr, const unsigned* r) {
  static_assert(NC == 4 || NC == 8 || NC == 12 || NC == 16 || NC == 32, "unsupported operand width");
  if (NC == 32) tmem_st32(taddr, r);
  else if (NC == 16) tmem_st16(taddr, r);
  else if (NC == 12) { tmem_st8(taddr, r); tmem_st4(taddr + 8, r + 8); }
  else if (NC == 8) tmem_st8(taddr, r);
  else tmem_st4(taddr, r);
}

// Stores v[0..NC) as operand columns [0, NC) (relative to the given addresses) of this thread's row: raw fp32 (the
// tensor core truncates to TF32) into A_hi and, in the split mode, the truncation remainder into A_lo.
template <int NC, int PASSES>
__device__ __forceinline__ void store_operand(unsigned t_hi, unsigned t_lo, const float* v, bool lo_pass) {
  unsigned r[NC];
#pragma unroll
  for (int i = 0; i < NC; ++i) r[i] = __float_as_uint(v[i]);
  tmem_st_n<NC>(t_hi, r);
  if (PASSES == 3 && lo_pass) {
#pragma unroll
    for (int i = 0; i < NC; i += 2) {   // remainder v - trunc(v): paired subtractions
      float a, b;
      up2(sub2(pk2(v[i], v[i + 1]), pk2(__uint_as_float(r[i] & 0xFFFFE000u), __uint_as_float(r[i + 1] & 0xFFFFE000u))), a, b);
      r[i] = __float_as_uint(a); r[i + 1] = __float_as_uint(b);
    }
    tmem_st_n<NC>(t_lo, r);
  }
}

template <int NC>
__device__ __forceinline__ void load_cols(unsigned taddr, float* v) {
  static_assert(NC == 16 || NC == 32, "unsupported load width");
  unsigned r[NC];
  if (NC == 32) tmem_ld32(taddr, r); else tmem_ld16(taddr, r);
  tmem_wait_ld();
#pragma unroll
  for (int i = 0; i < NC; ++i) v[i] = __uint_as_float(r[i]);
}

// One layer's MMA chain, fully unrolled over k-steps so that every descriptor is a constant offset (the chain then
// runs at the tensor-core floor of N/2 cycles per instruction, profiles/r1/tc_probe_b200.log).
template <int KS, int PASSES>
__device__ __forceinline__ void issue_chain(unsigned d, unsigned a_hi, unsigned a_lo, uint64_t b_hi, uint64_t b_lo, unsigned kb_stride16,
                                            unsigned idesc, unsigned first_acc, bool lo_pass) {
#pragma unroll
  for (int ks = 0; ks < KS; ++ks) {
    const uint64_t off = (uint64_t)((ks >> 2) * kb_stride16 + (ks & 3) * 2);
    mma_ts(d, a_hi + ks * 8, b_hi + off, idesc, ks > 0 ? 1u : first_acc);
    if (PASSES == 3) {
      if (lo_pass) mma_ts(d, a_lo + ks * 8, b_hi + off, idesc, 1u);
      mma_ts(d, a_hi + ks * 8, b_lo + off, idesc, 1u);
    }
  }
}

// 4-way partial sums: short dependency chains for the two warps that share an SM sub-partition.  Partial sums (a0, a1)
// and (a2, a3) are independent, so each pair is one paired instruction per step.
template <int N>
__device__ __forceinline__ float sum_n(const float* v) {
  f32x2 a01 = pk2(0.f, 0.f), a23 = pk2(0.f, 0.f);
#pragma unroll
  for (int i = 0; i < N; i += 4) { a01 = add2(a01, pk2(v[i], v[i + 1])); a23 = add2(a23, pk2(v[i + 2], v[i + 3])); }
  float a0, a1, a2, a3;
  up2(a01, a0, a1); up2(a23, a2, a3);
  return (a0 + a1) + (a2 + a3);
}
template <int N>
__device__ __forceinline__ float sumsq_centered_n(const float* v, float m) {
  const f32x2 mm = pk2(m, m);
  f32x2 a01 = pk2(0.f, 0.f), a23 = pk2(0.f, 0.f);
#pragma unroll
  for (int i = 0; i < N; i += 4) {
    const f32x2 d01 = sub2(pk2(v[i], v[i + 1]), mm), d23 = sub2(pk2(v[i + 2], v[i + 3]), mm);
    a01 = fma2(d01, d01, a01); a23 = fma2(d23, d23, a23);
  }
  float a0, a1, a2, a3;
  up2(a01, a0, a1); up2(a23, a2, a3);
  return (a0 + a1) + (a2 + a3);
}


__device__ __forceinline__ int perm64(int j, int d_read) { return j < d_read ? j : 32 + (j - d_read); }   // d_model vector -> X column
__device__ __forceinline__ int unperm64(int c, int d_read, int d_model) {   // X column -> d_model index or -1
  if (c < 32) return c < d_read ? c : -1;
  const int j = d_read + (c - 32);
  return j < d_model ? j : -1;
}

__device__ inline float tc_weight(const PmtModelDesc& D, const TcStep& o, const float* __restrict__ w, int n, int k) {
  const int DR = D.d_read, Dm = D.d_model, H = D.d_ffn / 2;
  switch (o.pk) {
    case PK_LINEAR: {
      const int nn = o.n_perm ? unperm64(n, DR, Dm) : (n < o.n_real ? n : -1);
      if (nn < 0) return 0.f;
      const float alpha = o.alpha_off >= 0 ? w[o.alpha_off] : 1.f;
      if (k == o.bias_col) return alpha * w[o.b_off + nn];
      const int kk = o.k_perm ? unperm64(k, DR, Dm) : (k < o.k_real ? k : -1);
      if (kk < 0) return 0.f;
      return alpha * (o.k_selu_scale ? SELU_SCALE : 1.f) * w[o.w_off + nn * o.k_real + kk];
    }
    case PK_PROJ1: {   // [ref set | alt set] side by side in N; LayerNorm affine folded (gated_mlp.py:185-187)
      const PmtBlockOffsets& BO = D.blocks[o.blk];
      const int set = n / NP1, c = n - set * NP1;
      // set layout: z1 (outputs 0..H) at columns 0..H), z2 (outputs H..2H) at columns 12..12+H)
      int nn = -1;
      if (c < H) nn = c;
      else if (c >= NP1 / 2 && c - NP1 / 2 < H) nn = H + (c - NP1 / 2);
      if (set > 1 || nn < 0) return 0.f;
      const int w_off = set ? BO.p1_alt_w : BO.p1_ref_w, b_off = set ? BO.p1_alt_b : BO.p1_ref_b;
      if (k == o.bias_col) {
        float acc = w[b_off + nn];
        for (int j = 0; j < Dm; ++j) acc = fmaf(w[w_off + nn * Dm + j], w[BO.ln_b + j], acc);
        return acc;
      }
      const int kk = unperm64(k, DR, Dm);
      if (kk < 0) return 0.f;
      return w[w_off + nn * Dm + kk] * w[BO.ln_w + kk];
    }
    case PK_PROJ2: {   // ref and alt sets stacked along K (gated_mlp.py:197-198)
      const PmtBlockOffsets& BO = D.blocks[o.blk];
      const int nn = unperm64(n, DR, Dm);
      if (nn < 0) return 0.f;
      // operand layout: [t_ref k 0..5 | t_alt k 0..5 | t_ref k 6..10 | t_alt k 6..10 | is_ref | is_alt]
      int unit = -1, set = 0;
      if (k < 6) { unit = k; set = 0; }
      else if (k < 12) { unit = k - 6; set = 1; }
      else if (k < 17) { unit = 6 + (k - 12); set = 0; }
      else if (k < 22) { unit = 6 + (k - 17); set = 1; }
      else if (k == 22) return w[BO.p2_ref_b + nn];
      else return w[BO.p2_alt_b + nn];
      if (unit >= H) return 0.f;
      return w[(set ? BO.p2_alt_w : BO.p2_ref_w) + nn * H + unit];
    }
    case PK_FINAL: {   // f = Q (W x + b + t): rotation and translation folded (euclidean_transformation.py:19-20)
      const int E = D.d_feat;
      if (n >= E) return 0.f;
      float acc = 0.f;
      if (k == o.bias_col) {
        for (int j = 0; j < E; ++j) acc = fmaf(w[D.rotation + n * E + j], w[o.b_off + j] + w[D.translation + j], acc);
        return acc;
      }
      const int kk = unperm64(k, DR, Dm);
      if (kk < 0) return 0.f;
      for (int j = 0; j < E; ++j) acc = fmaf(w[D.rotation + n * E + j], w[o.w_off + j * o.k_real + kk], acc);
      return acc;
    }
  }
  return 0.f;
}

// value of the backward's dY column nb of a proj1 step as a forward output column (-1: padding).  Backward layout:
// [half 0: ref z1 (6) | ref z2 (6) | alt z1 (6) | alt z2 (6)][half 1: the same for hidden units 6..11]
__host__ __device__ __forceinline__ int proj1_bwd_col(int nb, int H) {
  const int h = nb / 24, r = nb % 24, set = r / 12, z2 = (r % 12) / 6, unit = 6 * h + r % 6;
  if (unit >= H) return -1;
  return set * NP1 + (z2 ? NP1 / 2 + unit : unit);
}

}  // namespace tc
}  // namespace pmt

// host: the step program of the forward (pmt_tc.cu)
void pmt_tc_plan(const pmt::Plan& P, pmt::tc::TcPlan* out);
int pmt_launch_pack_tc(const pmt::Plan& P, const pmt::tc::TcPlan& T, const float* weights, unsigned char* image, cudaStream_t st);
int pmt_plan_tiles(const PmtBatch* batch, int max_variants, bool deterministic, int n_sm, int* tiles, int* claim_buf, int* n_claims_out,
                   cudaStream_t st);
