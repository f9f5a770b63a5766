// Declarations shared by the tensor-core haplotype-CNN forward (pmt_cnn_tc.cu) and the CNN backward that consumes the
// activations it saves (pmt_cnn_bwd.cu).
#pragma once
#include <cstring>

#include "pmt_host.h"
#include "pmt_tc_ptx.cuh"

namespace pmt {
namespace cnntc {

constexpr int EPI_WARPS = 16;
constexpr int THREADS = 32 * (EPI_WARPS + 1);
constexpr int MMA_WARP = EPI_WARPS;
constexpr int MAX_LAYERS = 10;
constexpr int MAX_CHUNKS = 4;
constexpr int CHUNK_COLS = 128;              // TMEM columns per chunk accumulator: [hi part N | lo part N]
constexpr int PLANE_ROWS = 344;
constexpr int PLANE_BYTES = PLANE_ROWS * 16;
constexpr int BUF_BYTES = 8 * PLANE_BYTES;   // one activation buffer: 32 channels
constexpr int C0 = 10;                       // one-hot channels: 2 haplotypes x 5 codes
constexpr int MAX_ITEMS = 24;                // (layer, chunk) work items per group
constexpr int MAX_TASKS = 8;                 // one-hot entries per lane in the im2col scatter

struct Layer {
  int first;      // im2col'd one-hot conv
  int taps;       // shifted-window convs: kernel size; first: number of input positions per row (ksize + dup)
  int ksteps;     // first: k-steps of 8 columns
  int N;          // output columns of the MMA (32, or 64 when dup)
  int dup, pool2; // fused MaxPool(2,1) after the first conv / MaxPool(2,2)
  int L_in, L_out, L_pool, L_next;
  int inv_L;      // ceil(65536 / L_in) + : row / L_in == (row * inv_L) >> 16 for rows < 512
  int act, to_global, out_ch;
  int to_tail;    // the split forward's last head layer: writes its pooled activation to the tail buffer
  int img_off, img_bytes;
  // packing
  int op, in_ch, ksize, flat_len, scale_in, is_linear;
};

struct Item {
  int layer, chunk;
  int need;   // index of the last done_bar this item's MMAs must have observed (0 = im2col, 1 + i = epilogue of item i)
};

struct Plan {
  int n_layers, n_items, G, L0, image_bytes;
  int smem;       // dynamic shared memory of hap_cnn_tc_kernel over these layers
  int n_chunks[MAX_LAYERS];
  Layer layer[MAX_LAYERS];
  Item item[MAX_ITEMS];
};

// ---- the split inference forward: hap_cnn_tc_kernel runs the head layers, hap_cnn_tail_kernel the short tail ----
// The tail is the trailing layers that each produce one position (after pooling), the first of them reading at most
// TAIL_MAX_K floats per variant and the others 32.  Every tail layer is a dense layer over its whole input window,
// M = 128 variants per tile: a conv's output positions sit side by side in N (N = 32 L_out) and a MaxPool(2, 2) that
// follows it is the max of the two column halves.  The head writes its last layer's pooled activation (selu_u applied)
// as fp32 to the tail buffer, [tile of 128 variants][K / 4 chunks][128 rows][4 floats]: the tail kernel's A operand in
// the no-swizzle K-major layout, so a K-stage of one tile is one contiguous bulk copy.
constexpr int TAIL_MAX_K = 256;
constexpr int MAX_TAIL = 3;
constexpr int TAIL_STAGE_CHUNKS = 8;                          // 16-byte K chunks per pipeline stage: 32 floats, 4 k-steps
constexpr int TAIL_PLANE = 128 * 16;                          // one K chunk of a 128-row tile
constexpr int TAIL_STAGE_BYTES = TAIL_STAGE_CHUNKS * TAIL_PLANE;
constexpr int TAIL_STAGES = 2;
constexpr int TAIL_EPI_WARPS = 8;                             // warps 0-7 epilogue, 8 MMA issuer, 9 bulk loader
constexpr int TAIL_THREADS = 32 * (TAIL_EPI_WARPS + 2);

struct TailPlan {
  int n_layers;
  int K0;              // floats per variant in the tail buffer: the first tail layer's input, L_in * 32
  int image_off;       // byte offset of the tail images inside the CNN image buffer (after the single kernel's)
  int image_bytes;
  int smem;            // dynamic shared memory of hap_cnn_tail_kernel
  Layer layer[MAX_TAIL];   // N = 32 L_out; img_off inside the tail images; to_global on the last
};

// ---- training: what the SAVE variant of the forward leaves in global memory for the backward (pmt_cnn_bwd.cu) ----
// Per group of G variants and per layer l that feeds another layer: the stored activation a_l = what the forward keeps in
// its shared-memory planes (bias added, pooled, selu_u applied: the SELU scale lives in the consuming weights) as
// [32 channels][G * L_next] floats, and -- for layers with a fused max-pool of two -- one byte per (channel group of 8,
// position) whose bit i tells that the SECOND element of the window won for channel 8 cg + i: [4][G * L_next] bytes.
struct SaveLayout {
  int G, n_layers;
  int group_floats;             // floats per group
  int a_off[MAX_LAYERS];        // float offset of a_l inside a group (-1: not saved)
  int bits_off[MAX_LAYERS];     // float offset of the window bits (-1: no pool)
};

}  // namespace cnntc

// the tensor-core CNN backward's plan (pmt_cnn_bwd.cu)
namespace cnnbwd {

constexpr int THREADS = 512, WARPS = THREADS / 32;
constexpr int MAXL = cnntc::MAX_LAYERS;
constexpr int NT = 4;            // n-tiles of 8 columns per weight-gradient unit
constexpr int SLOTS = 3;         // weight-gradient units per warp
constexpr int MAX_UNITS = SLOTS * WARPS;
constexpr int MAX_NPV = 4;       // data gradient: n-tiles of 8 input positions per variant

struct BLayer {
  int Cin, Cout, ks, L_in, L_out, L_pool;
  int dup, pool2, selu, first, to_global, is_linear, flat_len;
  int w_off, b_off, op_in_ch;
  int Cin8, Cout8, Mt_w, Mt_d, kpv, npv;
  int lm, lpg, ldy;        // dY_l: left margin (ks - 1), per-variant stride, row stride (floats)
  int ld_a, a_smem;        // INPUT plane a_{l-1} in shared memory: row stride, float offset (l > 0)
  int ld_g;                // row stride of g_{l-1}, the data gradient this layer produces (l > 0)
  int img_off;             // float offset of the data-gradient image inside the image buffer
  int save_in, save_bits;  // float offsets inside a group's save block: a_{l-1}; this layer's window bits (-1: none)
  int bits_smem;           // byte offset of this layer's window bits in shared memory
  int inv_vt_pad_;
  float s_in;              // SELU scale of the previous layer (folded into the forward's weight images): a_{l-1} = s_in * saved
};
struct Unit { int layer, m, nt0, cnt; };
struct BPlan {
  int n_layers, VT, G, n_units, group_floats;
  int img_total, a_total, dy_floats, g_floats, bits_bytes, codes_stride, L0;
  int inv_vt;              // ceil(65536 / VT): pair / VT == (pair * inv_vt) >> 16 for pair < 1024
  int smem_bytes;
  BLayer layer[MAXL];
  Unit unit[MAX_UNITS];
};

}  // namespace cnnbwd
}  // namespace pmt

// host (pmt_cnn_tc.cu)
bool pmt_build_cnn_tc_plan(const pmt::Plan& P, pmt::cnntc::Plan* out);
// The head + tail pair of the inference forward from the single kernel's plan; false when the CNN has no tail.
bool pmt_build_cnn_split_plan(const pmt::cnntc::Plan& T, int hap_len, pmt::cnntc::Plan* head, pmt::cnntc::TailPlan* tail);
void pmt_cnn_save_layout(const pmt::cnntc::Plan& T, pmt::cnntc::SaveLayout* out);
int pmt_pack_cnn_tc_images(const pmt::Plan& P, const pmt::cnntc::Plan& T, const float* weights, unsigned char* image, cudaStream_t st);
// the forward over variants [v_first, v_first + n) of the batch with every layer's activations saved; `image` must hold
// the packed weight images (pmt_launch_cnn_tc with reuse_image = false packs them)
int pmt_launch_cnn_tc_save(const pmt::Plan& P, const pmt::cnntc::Plan& T, const float* weights, const PmtBatch* batch, int v_first, int n,
                           float* info_seq, const unsigned char* image, float* save, int n_sm, cudaStream_t st);
