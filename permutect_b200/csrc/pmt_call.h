// The call plan: which kernels one C-ABI call of the model (pmt_workspace_size, pmt_train_saved_bytes,
// pmt_backward_kernels, pmt_forward, pmt_forward_prepared, pmt_forward_train, pmt_backward) runs, with what launch geometry,
// and where their buffers live.  pmt_call_plan decides all of it once per call from the model, the batch, the precision
// mode, the device and the test and measurement overrides (read_overrides in pmt_forward.cu, its only reader): the kernels,
// the tile planner, the pass count, the claim sizes and grids of the SIMT kernels, every kernel's dynamic shared memory and
// weight-ring stages, and the maps of the forward workspace, the backward workspace and the saved-forward buffer
// (pmt_call.cu, which also resolves them against a caller's buffer).  It also decides whether the forward or the backward
// would be refused (fwd_refusal, bwd_refusal); the entry points check that, and resolve their buffers, before their first
// CUDA call, so a refused call leaves the caller's buffers untouched.  The launchers take their plans, grids and pointers
// from it and decide nothing again.
#pragma once
#include "pmt_cnn_tc.cuh"
#include "pmt_tc.cuh"

// Kernels that keep one private buffer of partial sums per CTA (the SIMT backward, the tensor-core backward's slots, the
// SIMT long-set scratch) size those buffers for this many CTAs and cap their grids at it.
constexpr int PMT_PARTIAL_CTAS = 148;

// The batch's row count, or 16 rows per variant when the caller did not give one.
inline long long pmt_row_hint(const PmtBatch* batch) { return batch->n_rows > 0 ? batch->n_rows : 16LL * batch->n_variants; }

// Grid of a tile kernel: the tile count is only known on the device, so it is estimated from the row hint (a tile holds
// ~110 rows of whole variants) plus one partial tile per planner claim; one CTA per tile until every SM has one.
inline int pmt_tile_grid(const PmtBatch* batch, int n_claims, int n_sm) {
  long long est_tiles = pmt_row_hint(batch) / 100 + n_claims;
  if (est_tiles > batch->n_variants) est_tiles = batch->n_variants;
  const int grid = est_tiles < n_sm ? (int)est_tiles : n_sm;
  return grid < 1 ? 1 : grid;
}

// Variants per recompute + backward pass of the tensor-core haplotype-CNN backward: bounds the saved activations of a
// pass (5.3 KB per variant).
constexpr int PMT_CNN_BWD_CHUNK = 65536;

// Variants per claim of the tile planner and the bytes of its per-claim scratch (pmt_tc.cu).
int pmt_plan_claim_variants(int n_variants, int n_sm);
size_t pmt_plan_claim_bytes(int n_variants, int n_sm);

namespace pmt {

enum class InfoKernel { WARP, ROWS, TILE };     // info_mlp_warp_kernel (small batches), info_mlp_rows_kernel<W4>, info_mlp_kernel
// hap_cnn_tc_kernel over every layer, the head + tail pair (hap_cnn_tc_kernel over the head layers, then
// hap_cnn_tail_kernel), the SAVE variant of the first (training forward), hap_cnn_kernel
enum class CnnKernel { TC, TC_TAIL, TC_SAVE, SIMT };
enum class ReadsKernel { TC, TC_SAVE, SIMT };   // reads_forward_tc_kernel, its SAVE variant (training forward), reads_forward_kernel
enum class LongKernel { NONE, TC, SIMT };       // sets longer than a tile: reads_forward_tc_kernel<.., LONG>, reads_forward_long_kernel

// The maps of a call's buffers (pmt_call.cu).  A region is `bytes` at byte offset `off`; a region that a kernel needs at
// an aligned address lies in a slot with the slack to realign it as an absolute address (the C-ABI does not require an
// aligned workspace), and the regions inside such a slot are offsets from its aligned start.

struct Region {
  size_t off, bytes;
};

// The long-set region of the tensor-core forward (reads_forward_tc_kernel<.., LONG>), from its 256-aligned start.
// counters: the arrival counters mf_cnt and fin_cnt, zeroed together.
struct LongLayout {
  int cap, max_tiles, R;
  Region list, n_tiles, tiles, counters, fin_cnt, mf_part, fin_part;
  size_t bytes;
};

// The tensor-core backward's region of the backward workspace (pmt_tc_bwd.cu), from its 1024-aligned start.
struct BwdLayout {
  Region image_f, image_t, tiles, claims, partials, reduced, scratch;
  size_t total;
  int chunk_tiles, n_chunks, n_claims;
};

// The buffer pmt_forward_train fills for pmt_backward, from its base (256-byte aligned): [256 bytes, unused][tile list]
// [operand scratch of every tile of the deterministic list][haplotype-CNN activations].  The tile count is only known on
// the device, so the scratch is sized for the bound.  total == 0: no saved forward for this call.
struct SavedLayout {
  Region tiles, scratch, cnn;
  size_t total;
  long long bound;
};

// The forward workspace (pmt_forward, pmt_forward_prepared, pmt_forward_train).  The weight images sit at FIXED offsets
// (they depend on the model only: pmt_forward_prepared finds them there), the batch-dependent regions follow:
//   [256 B counters][SIMT images][tcgen05 read-kernel images][tcgen05 CNN images] | [info_seq][long-set scratch]
//   [tile slot][long-set tensor-core slot][CNN tail buffer]
// tc_image is realigned to 1024 bytes.  The tile slot (realigned to 256) holds the inference tile list with the packed
// planner's variant order after it, or the training forward's planner claims.
struct FwdMap {
  Region counters, image, tc_image, cnn_tc_image, info_seq, long_scratch, cnn_tail;
  size_t tile_slot, long_slot;   // long_slot: LongLayout (C.long_tc), realigned to 256
  Region tiles, perm, claims;    // in the tile slot
  size_t long_scratch_floats;    // LongKernel::SIMT: per CTA
  size_t end;
};

// The backward workspace (pmt_backward):
//   [256 B][SIMT images][partials][activation scratch][info_seq][d_info_seq] | [long-set scratch]
//   [tensor-core read-path slot][tensor-core CNN slot]
// The read-path slot holds BwdLayout (C.tc_bwd) from its 1024-aligned start; the CNN slot, realigned to 256, holds the
// forward weight images of the recompute, the data-gradient images and the saved activations of one chunk.
struct BwdMap {
  Region image, partials, scratch, info_seq, d_info_seq, long_scratch;
  size_t tc_slot, cnn_slot;
  Region cnn_fwd_image, cnn_bwd_image, cnn_save;   // in the CNN slot
  size_t scr_floats, long_floats;                  // per CTA: the activation scratch, the long-set scratch
  int long_grid;                                   // reads_backward_long_kernel (0: no long sets)
  size_t end;
};

// A tensor-core kernel's weight ring: n_stages stages of stage_bytes next to its fixed carve, `smem` dynamic bytes in all.
// n_stages < 2: the ring does not fit.
struct Ring {
  int stage_bytes, n_stages;
  size_t smem;
};

// The SIMT haplotype-CNN backward (hap_cnn_backward_kernel, pmt_backward.cu): vt variants per pass; every layer's
// activation of the pass stays in shared memory, channel-major with a per-variant stride lp[i] (multiple of 4) and a
// channel stride ld[i] == 4 (mod 32).
struct CnnBwdGeom {
  int vt, n_spatial, n_linear, vs;
  int ch[PMT_MAX_CNN_OPS + 1], len[PMT_MAX_CNN_OPS + 1], lp[PMT_MAX_CNN_OPS + 1], ld[PMT_MAX_CNN_OPS + 1];
  int act_off[PMT_MAX_CNN_OPS + 1];   // activation entering spatial op i ([n_spatial] = last output)
  int lpg[PMT_MAX_CNN_OPS], ldg[PMT_MAX_CNN_OPS];   // zero-padded layout of conv op i's output gradient
  int act_total, gbuf_floats, stage_floats;
};

// A SIMT kernel that claims variants from a counter: `claim` variants per claim, `grid` CTAs.
struct Claims {
  int claim, n_claims, grid;
};

struct CallPlan {
  Plan P;
  CnnGeom G;
  int mode;                    // PMT_PRECISION_*
  int passes;                  // MMA passes of the tensor-core inference kernels: 1 in PMT_PRECISION_TF32, 3 (split TF32) else
  int n_sm;
  // why pmt_forward / pmt_forward_prepared / pmt_forward_train, and why pmt_backward, would be refused ("": they run)
  char fwd_refusal[160], bwd_refusal[160];
  bool reads_tc_ok;            // the model is inside the envelope of the tensor-core read kernels
  bool cnn_tc_ok, cnn_bwd_ok;  // ... of the tensor-core haplotype CNN forward, and of its backward
  tc::TcPlan T;                // step program of the read path (built for every model: its image is part of the layout)
  cnntc::Plan C;               // cnn_tc_ok
  bool cnn_split;              // cnn_tc_ok and the CNN has a tail: CH + CT are planned
  cnntc::Plan CH;              // cnn_split: the head layers
  cnntc::TailPlan CT;          // cnn_split: the tail layers
  cnnbwd::BPlan CB;            // cnn_bwd_ok
  // forward
  InfoKernel info;
  int info_w4;                 // InfoKernel::ROWS: the template width
  size_t info_smem;            // ... and the dynamic shared memory of the info MLP kernel `info`
  CnnKernel cnn;
  size_t cnn_simt_smem;        // hap_cnn_kernel (the CNN forward of CnnKernel::SIMT and of the backward's recompute)
  ReadsKernel reads;
  bool packed_planner;         // ReadsKernel::TC: plan_tiles_packed_kernel; else the sequential planner (pmt_plan_tiles)
  Ring ring;                   // reads_forward_tc_kernel<passes, false, *> (inference, and the long-set tiles)
  Ring ring_save;              // reads_forward_tc_kernel<3, true, false> (training forward, the backward's recompute)
  size_t reads_smem;           // reads_forward_kernel and reads_forward_long_kernel
  Claims fwd_claims;           // reads_forward_kernel (batch given)
  int fwd_long_grid;           // reads_forward_long_kernel (batch given)
  LongKernel lng;
  bool simt_gemm, simt_conv;   // SIMT weight images of the tile GEMMs / the convolutions that the batch-independent kernels read
  LongLayout long_tc;          // lng == LongKernel::TC
  SavedLayout saved;           // saved.total > 0: the saved training forward exists
  FwdMap fwd;
  // backward
  bool bwd_reads_tc, bwd_cnn_tc;
  BwdLayout tc_bwd;            // reads_tc_ok
  Ring ring_bwd;               // reads_backward_tc_kernel
  size_t bwd_smem;             // reads_backward_kernel and reads_backward_long_kernel
  size_t info_bwd_smem;        // info_mlp_backward_kernel
  Claims bwd_claims;           // reads_backward_kernel (batch given)
  CnnBwdGeom cnn_bwd;          // !bwd_cnn_tc: hap_cnn_backward_kernel's geometry ...
  size_t cnn_bwd_smem;         // ... and dynamic shared memory
  BwdMap bwd;
};

// The maps resolved against a caller's buffer: typed pointers to every region (pmt_forward_buffers, pmt_backward_buffers,
// pmt_saved_buffers).
struct LongBuffers {
  int *list, *n_tiles;
  tc::LongTile* tiles;
  int *counters, *fin_cnt;   // counters: mf_cnt, and the start of what the launcher zeroes
  float *mf_part, *fin_part;
};
struct FwdBuffers {
  int* counters;
  float* image;
  unsigned char *tc_image, *cnn_tc_image;
  float *info_seq, *long_scratch;
  int *tiles, *perm, *claims;   // perm: NULL unless the packed planner runs
  LongBuffers lng;
  float* cnn_tail;
};
struct TcBwdBuffers {
  unsigned char *image_f, *image_t;
  int *tiles, *claims;
  float *partials, *reduced;
  unsigned char* scratch;
};
struct CnnBwdBuffers {
  unsigned char* fwd_image;
  float *bwd_image, *save;
};
struct BwdBuffers {
  float *image, *partials, *scratch, *info_seq, *d_info_seq, *long_scratch;
  TcBwdBuffers tc;
  CnnBwdBuffers cnn;
};
struct SavedBuffers {
  int* tiles;
  unsigned char* scratch;
  float* cnn;
};

}  // namespace pmt

int pmt_sm_count();
// `train`: the call is pmt_forward_train (its CNN and read kernels are the SAVE variants).  `batch` may be NULL (a size
// query without a batch).
int pmt_call_plan(const PmtModelDesc* desc, const PmtBatch* batch, bool train, pmt::CallPlan* out);

// pmt_call.cu: the maps of pmt_call_plan -- the saved-forward buffer (before the kernels are chosen: a call without one
// runs no SAVE kernel), the long-set tensor-core region (false: that path is not available for this batch, the FP32
// long-set kernel takes the long sets), the tensor-core backward's region (`max_chunk_tiles` >= 1: at most that many tiles
// per recompute + backward pass, else the default), then the two workspaces (once every kernel is chosen)
pmt::SavedLayout pmt_saved_layout(const pmt::CallPlan& C, const PmtBatch* batch);
bool pmt_tc_long_layout(const pmt::Plan& P, const PmtBatch* batch, int n_sm, pmt::LongLayout* L);
pmt::BwdLayout pmt_tc_bwd_layout(const pmt::tc::TcPlan& T, const PmtBatch* batch, int max_chunk_tiles);
void pmt_plan_workspaces(pmt::CallPlan& C, const PmtBatch* batch);
// The resolvers: the maps laid over a caller's buffer of `bytes` bytes.  1 (error set): the buffer is too small.
int pmt_forward_buffers(const pmt::CallPlan& C, void* workspace, size_t bytes, pmt::FwdBuffers* out);
int pmt_backward_buffers(const pmt::CallPlan& C, void* workspace, size_t bytes, pmt::BwdBuffers* out);
int pmt_saved_buffers(const pmt::CallPlan& C, const void* saved, size_t bytes, pmt::SavedBuffers* out);

// pmt_forward.cu: the per-variant embeddings and the SIMT weight images (gemm: the tile GEMMs of the read path, the info MLP
// and their backward; conv: the SIMT haplotype CNN and its backward)
int pmt_launch_prepare(const pmt::CallPlan& C, const float* weights, float* image, cudaStream_t st, bool gemm, bool conv);
int pmt_launch_info_mlp(const pmt::CallPlan& C, const float* weights, const float* image, const PmtBatch* batch, float* info_seq,
                        cudaStream_t st);
int pmt_launch_hap_cnn_simt(const pmt::CallPlan& C, const float* weights, const float* image, const PmtBatch* batch, float* info_seq,
                            cudaStream_t st);
// pmt_backward.cu
// the SIMT backward's shared memory, claims and CNN geometry, and bwd_refusal for them (pmt_call_plan, once
// bwd_reads_tc and bwd_cnn_tc are decided)
void pmt_plan_backward(pmt::CallPlan& C, const PmtBatch* batch);
// pmt_tc.cu
bool pmt_tc_supported(const pmt::Plan& P);
pmt::Ring pmt_tc_ring(const pmt::tc::TcPlan& T, int passes);
int pmt_launch_reads_tc(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                        const pmt::FwdBuffers& W, bool reuse_images, cudaStream_t st);
int pmt_launch_reads_tc_long(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                             const pmt::FwdBuffers& W, cudaStream_t st);
// pmt_tc_bwd.cu
// the most tiles the deterministic training tile list of `batch` can hold (planned in `n_claims` claims)
long long pmt_train_tile_bound(const PmtBatch* batch, int n_claims);
pmt::Ring pmt_tc_bwd_ring(const pmt::tc::TcPlan& T);
int pmt_launch_reads_tc_save(const pmt::CallPlan& C, const pmt::tc::TcArgs& A, int grid, cudaStream_t st);
int pmt_tc_forward_train(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                         const pmt::FwdBuffers& W, const pmt::SavedBuffers& S, cudaStream_t st);
// `saved`: NULL, or what pmt_forward_train saved for this batch
int pmt_launch_reads_tc_backward(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, const float* info_seq,
                                 const float* d_logits_bk, const float* d_alt_means, const float* d_ref_means, float* d_info_seq,
                                 const pmt::TcBwdBuffers& W, int* grid_out, cudaStream_t st, const pmt::SavedBuffers* saved);
int pmt_finish_reads_tc_backward(const pmt::CallPlan& C, const float* weights, float* d_weights, const pmt::TcBwdBuffers& W, int grid,
                                 cudaStream_t st);
// pmt_cnn_tc.cu
size_t pmt_cnn_tc_image_bytes(const pmt::CallPlan& C);
// C.cnn TC or TC_TAIL; the images of both are packed unless reuse_image
int pmt_launch_cnn_tc(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq, const pmt::FwdBuffers& W,
                      bool reuse_image, cudaStream_t st);
// pmt_cnn_bwd.cu
bool pmt_build_cnn_bwd_plan(const pmt::Plan& P, const pmt::cnntc::Plan& T, pmt::cnnbwd::BPlan* out);
int pmt_cnn_forward_train(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq, unsigned char* image,
                          float* save, cudaStream_t st);
// `saved`: NULL, or the CNN activations pmt_forward_train saved for this batch
int pmt_launch_cnn_backward_mma(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq,
                                const float* d_info_seq, float* partials, const pmt::CnnBwdBuffers& W, cudaStream_t st,
                                const float* saved);
