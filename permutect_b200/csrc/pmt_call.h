// The call plan: which kernels one C-ABI call of the model (pmt_workspace_size, pmt_train_saved_bytes,
// pmt_backward_kernels, pmt_forward, pmt_forward_prepared, pmt_forward_train, pmt_backward) runs, with what launch geometry,
// and where their buffers live.  pmt_call_plan decides all of it once per call from the model, the batch, the precision
// mode, the device and the test and measurement overrides (read_overrides in pmt_forward.cu, its only reader): the kernels,
// the tile planner, the pass count, the claim sizes and grids of the SIMT kernels, every kernel's dynamic shared memory and
// weight-ring stages.  It also decides whether the forward or the backward would be refused (fwd_refusal, bwd_refusal);
// the entry points check that before their first CUDA call, so a refused call leaves the caller's buffers untouched.  The
// launchers take their plans, grids and regions from it and decide nothing again.
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

// A tile list: [0] = count, (first variant, variants) pairs from [2].
inline size_t pmt_tile_list_bytes(int n_variants) { return ((size_t)(2 + 2 * (size_t)n_variants) * sizeof(int) + 255) & ~(size_t)255; }

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

// The long-set region of the tensor-core forward (pmt_tc.cu), byte offsets from its 256-aligned base.
struct LongLayout {
  int cap, max_tiles, R;
  size_t list, n_tiles, tiles, counters, counters_bytes, fin_cnt, mf_part, fin_part, end;
};

// The tensor-core backward's region of the backward workspace (pmt_tc_bwd.cu), byte offsets from its 1024-aligned base.
struct BwdLayout {
  size_t image_f, image_t, tiles, claims, partials, reduced, scratch, total;
  int chunk_tiles, n_chunks, n_claims;
};

// The buffer pmt_forward_train fills for pmt_backward: [256-byte header][tile list][operand scratch of every tile of the
// deterministic list][haplotype-CNN activations].  The tile count is only known on the device, so the scratch is sized for
// the bound.  total == 0: no saved forward for this call.
struct SavedLayout {
  size_t tiles, scratch, cnn, total;
  long long bound;
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
  // backward
  bool bwd_reads_tc, bwd_cnn_tc;
  BwdLayout tc_bwd;            // reads_tc_ok
  Ring ring_bwd;               // reads_backward_tc_kernel
  size_t bwd_smem;             // reads_backward_kernel and reads_backward_long_kernel
  size_t info_bwd_smem;        // info_mlp_backward_kernel
  Claims bwd_claims;           // reads_backward_kernel (batch given)
  CnnBwdGeom cnn_bwd;          // !bwd_cnn_tc: hap_cnn_backward_kernel's geometry ...
  size_t cnn_bwd_smem;         // ... and dynamic shared memory
};

}  // namespace pmt

int pmt_sm_count();
// `train`: the call is pmt_forward_train (its CNN and read kernels are the SAVE variants).  `batch` may be NULL (a size
// query without a batch).
int pmt_call_plan(const PmtModelDesc* desc, const PmtBatch* batch, bool train, pmt::CallPlan* out);

// pmt_forward.cu: the per-variant embeddings and the SIMT weight images (gemm: the tile GEMMs of the read path, the info MLP
// and their backward; conv: the SIMT haplotype CNN and its backward)
int pmt_launch_prepare(const pmt::CallPlan& C, const float* weights, float* image, cudaStream_t st, bool gemm, bool conv);
int pmt_launch_info_mlp(const pmt::CallPlan& C, const float* weights, const float* image, const PmtBatch* batch, float* info_seq,
                        cudaStream_t st);
int pmt_launch_hap_cnn_simt(const pmt::CallPlan& C, const float* weights, const float* image, const PmtBatch* batch, float* info_seq,
                            cudaStream_t st);
// pmt_backward.cu
size_t pmt_backward_workspace_size(const pmt::CallPlan& C, const PmtBatch* batch);
// the SIMT backward's shared memory, claims and CNN geometry, and bwd_refusal for them (pmt_call_plan, once
// bwd_reads_tc and bwd_cnn_tc are decided)
void pmt_plan_backward(pmt::CallPlan& C, const PmtBatch* batch);
// pmt_tc.cu
bool pmt_tc_supported(const pmt::Plan& P);
bool pmt_tc_long_layout(const pmt::Plan& P, const PmtBatch* batch, int n_sm, pmt::LongLayout* L);
size_t pmt_tc_tiles_bytes(int n_variants);
pmt::Ring pmt_tc_ring(const pmt::tc::TcPlan& T, int passes);
int pmt_launch_reads_tc(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                        unsigned char* image_buf, unsigned char* tiles_buf, bool reuse_images, cudaStream_t st);
int pmt_launch_reads_tc_long(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                             unsigned char* image_buf, unsigned char* long_buf, cudaStream_t st);
// pmt_tc_bwd.cu
// `max_chunk_tiles` >= 1: at most that many tiles per recompute + backward pass (else the default)
pmt::BwdLayout pmt_tc_bwd_layout(const pmt::tc::TcPlan& T, const PmtBatch* batch, int max_chunk_tiles);
pmt::Ring pmt_tc_bwd_ring(const pmt::tc::TcPlan& T);
int pmt_launch_reads_tc_save(const pmt::CallPlan& C, const pmt::tc::TcArgs& A, int grid, cudaStream_t st);
pmt::SavedLayout pmt_saved_layout(const pmt::CallPlan& C, const PmtBatch* batch);
int pmt_tc_forward_train(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, const PmtOutputs* out,
                         unsigned char* image_buf, unsigned char* claim_buf, unsigned char* saved, cudaStream_t st);
int pmt_launch_reads_tc_backward(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, const float* info_seq,
                                 const float* d_logits_bk, const float* d_alt_means, const float* d_ref_means, float* d_info_seq,
                                 unsigned char* ws, size_t ws_bytes, int* grid_out, cudaStream_t st, const unsigned char* saved);
int pmt_finish_reads_tc_backward(const pmt::CallPlan& C, const float* weights, float* d_weights, unsigned char* ws, int grid,
                                 cudaStream_t st);
// pmt_cnn_tc.cu
size_t pmt_cnn_tc_image_bytes(const pmt::CallPlan& C);
size_t pmt_cnn_tail_buffer_bytes(const pmt::CallPlan& C, int n_variants);
// C.cnn TC or TC_TAIL (`tail_buf`: pmt_cnn_tail_buffer_bytes, 16-byte aligned); the images of both are packed unless reuse_image
int pmt_launch_cnn_tc(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq, unsigned char* image,
                      bool reuse_image, float* tail_buf, cudaStream_t st);
// pmt_cnn_bwd.cu
bool pmt_build_cnn_bwd_plan(const pmt::Plan& P, const pmt::cnntc::Plan& T, pmt::cnnbwd::BPlan* out);
size_t pmt_cnn_bwd_workspace_bytes(const pmt::CallPlan& C, const PmtBatch* batch);
int pmt_cnn_forward_train(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq, unsigned char* image,
                          float* save, cudaStream_t st);
int pmt_launch_cnn_backward_mma(const pmt::CallPlan& C, const float* weights, const PmtBatch* batch, float* info_seq,
                                const float* d_info_seq, float* partials, unsigned char* ws, size_t ws_bytes, cudaStream_t st,
                                const float* saved);
