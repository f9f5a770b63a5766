// Where every byte of a model call lives: the maps of the forward workspace, the backward workspace and the saved-forward
// buffer that pmt_call_plan puts in the call plan (pmt_call.h), the size queries that report them, and the resolvers that
// lay them over a caller's buffer.  The resolvers are the only code that aligns a pointer into a caller's buffer of a model
// call; every offset, alignment and slack they rely on is set here.
#include <algorithm>

#include "pmt_call.h"

using namespace pmt;
using namespace pmt::tc;

static size_t align_to(size_t n, size_t a) { return (n + a - 1) & ~(a - 1); }

// A tile list: [0] = count, (first variant, variants) pairs from [2].
static size_t tile_list_bytes(int n_variants) { return align_to((2 + 2 * (size_t)n_variants) * sizeof(int), 256); }
// the packed planner's variant order
static size_t perm_bytes(int n_variants) { return align_to((size_t)n_variants * sizeof(int), 256); }

// ---- the saved-forward buffer and the tensor-core regions ----

// Tiles per recompute / backward pass: bounds the operand scratch (0.7 MB per tile: 5.9 GB).  The scratch is streamed through
// HBM either way (it never was L2-sized), so fewer, longer passes only save launches -- the tile bound is an upper bound and most
// passes beyond the first found nothing to do -- and the partly filled last round of every pass.
static const int kChunkTiles = 8192;
// measured: 9 GB (65 536 variants) wins 14 %, 27 GB (200 000) loses to the recompute
static const size_t kTrainSavedBudget = (size_t)16 << 30;

// claims of the training tile list (planned with PMT_PARTIAL_CTAS for the SM count, whatever the device)
static int train_claims(int n_variants) {
  const int cv = pmt_plan_claim_variants(n_variants, PMT_PARTIAL_CTAS);
  return n_variants > 0 ? (n_variants + cv - 1) / cv : 0;
}

SavedLayout pmt_saved_layout(const CallPlan& C, const PmtBatch* batch) {
  SavedLayout S;
  memset(&S, 0, sizeof(S));
  if (C.mode != PMT_PRECISION_TF32X3 || !batch || batch->n_variants <= 0 || !C.bwd_reads_tc || !C.bwd_cnn_tc) return S;
  const int B = batch->n_variants;
  S.bound = pmt_train_tile_bound(batch, train_claims(B));
  S.tiles = {256, tile_list_bytes(B)};
  S.scratch = {align_to(S.tiles.off + S.tiles.bytes + 256, 1024), (size_t)S.bound * C.T.tile_bytes};
  S.cnn = {align_to(S.scratch.off + S.scratch.bytes + 1024, 1024), ((size_t)B + C.C.G - 1) / C.C.G * C.CB.group_floats * sizeof(float)};
  const size_t total = S.cnn.off + S.cnn.bytes + 256 + 1024;
  if (total <= kTrainSavedBudget) S.total = total;
  return S;
}

// false: the long-set tensor-core path is not available for this batch (no long sets, unknown row count, or a set longer
// than one round of tiles) -- the FP32 long-set kernel takes them.
bool pmt_tc_long_layout(const Plan& P, const PmtBatch* batch, int n_sm, LongLayout* L) {
  if (!batch || !pmt_has_long_sets(batch) || batch->n_rows <= 0 || !pmt_tc_supported(P)) return false;
  const int R = 2 * n_sm;
  const long long t_max = (batch->max_rows_per_variant + TILE - 1) / TILE + 1;        // ceil per side
  if (t_max > R) return false;
  long long cap = batch->n_rows / (TILE - 2);
  if (cap > batch->n_variants) cap = batch->n_variants;
  if (cap < 1) cap = 1;
  const long long sum_t = batch->n_rows / TILE + 2 * cap;
  const long long rounds = sum_t / (R - t_max + 1) + 1;
  const long long max_tiles = sum_t + rounds * (t_max - 1) + R;
  if (max_tiles > 0x3fffffff) return false;
  L->cap = (int)cap; L->max_tiles = (int)max_tiles; L->R = R;
  size_t off = 0;
  auto take = [&](size_t bytes) { const Region r = {off, bytes}; off += align_to(bytes, 256); return r; };
  L->list = take((size_t)(1 + cap) * sizeof(int));
  L->n_tiles = take(256);
  L->tiles = take((size_t)max_tiles * sizeof(LongTile));
  const Region mf_cnt = take((size_t)max_tiles * P.d.n_blocks * sizeof(int));
  L->fin_cnt = take((size_t)max_tiles * sizeof(int));
  L->counters = {mf_cnt.off, off - mf_cnt.off};
  L->mf_part = take((size_t)max_tiles * P.d.n_blocks * MAXH * sizeof(float));
  L->fin_part = take((size_t)max_tiles * LONG_FIN_W * sizeof(float));
  L->bytes = off;
  return true;
}

BwdLayout pmt_tc_bwd_layout(const TcPlan& T, const PmtBatch* batch, int max_chunk_tiles) {
  BwdLayout L;
  memset(&L, 0, sizeof(L));
  const int B = batch ? batch->n_variants : 0;
  size_t off = 1024;
  L.image_f = {off, (size_t)T.image_bytes}; off += L.image_f.bytes + 2048;
  L.image_t = {off, (size_t)T.t_image_bytes}; off += L.image_t.bytes + 2048;
  L.tiles = {off, tile_list_bytes(B)}; off += L.tiles.bytes + 256;
  L.claims = {off, pmt_plan_claim_bytes(B, PMT_PARTIAL_CTAS)}; off += L.claims.bytes + 256;
  L.partials = {off, (size_t)2 * PMT_PARTIAL_CTAS * T.part_floats * sizeof(float)}; off += L.partials.bytes;
  L.reduced = {off, (size_t)T.part_floats * sizeof(float)}; off += L.reduced.bytes + 256;
  off = align_to(off, 1024);
  L.n_claims = train_claims(B);
  const long long bound = batch ? pmt_train_tile_bound(batch, L.n_claims) : 1;
  const int chunk_cap = max_chunk_tiles >= 1 ? max_chunk_tiles : kChunkTiles;
  L.chunk_tiles = (int)(bound < chunk_cap ? bound : chunk_cap);
  L.n_chunks = (int)((bound + L.chunk_tiles - 1) / L.chunk_tiles);
  L.scratch = {off, (size_t)L.chunk_tiles * T.tile_bytes};
  L.total = off + L.scratch.bytes + 1024;
  return L;
}

// ---- the workspaces ----

// long-set scratch of the FP32 forward kernel: per CTA, one (x, z) image pair per chunk of the longest variant
static size_t long_scratch_floats_per_cta(const Plan& P, const PmtBatch* batch) {
  const size_t chunks = (size_t)((batch->max_rows_per_variant + 3 + TILE - 1) / TILE) + 1;
  return chunks * (size_t)(P.d.d_model + P.d.d_ffn) * LD;
}

// The CNN tail buffer is sized whenever the CNN has a tail and inference runs a tensor-core CNN, even where the plan chose
// the single kernel: sizing for C.cnn == TC_TAIL alone would shrink pmt_workspace_size below the pair's batch-size
// threshold, and the sizes the library reports stay as they were.
static size_t cnn_tail_bytes(const CallPlan& C, int n_variants) {
  const bool tc = C.cnn == CnnKernel::TC || C.cnn == CnnKernel::TC_TAIL;
  return C.cnn_split && tc ? (size_t)(n_variants + 127) / 128 * 128 * C.CT.K0 * sizeof(float) : 0;
}

static FwdMap forward_map(const CallPlan& C, const PmtBatch* batch) {
  const int B = batch ? batch->n_variants : 0;
  FwdMap M;
  memset(&M, 0, sizeof(M));
  M.counters = {0, 256};
  size_t off = 256;
  M.image = {off, pmt_image_bytes(C.P, C.G)};
  off = align_to(off + M.image.bytes, 1024);
  M.tc_image = {off, (size_t)C.T.image_bytes};   // + slack to realign to 1024
  off = align_to(off + M.tc_image.bytes + 2048, 256);
  M.cnn_tc_image = {off, pmt_cnn_tc_image_bytes(C)};
  off = align_to(off + M.cnn_tc_image.bytes, 256);
  M.info_seq = {off, (size_t)B * (C.P.d.d_info + C.P.d.d_seq) * sizeof(float)};
  off = align_to(off + M.info_seq.bytes, 256);
  if (C.lng == LongKernel::SIMT) M.long_scratch_floats = long_scratch_floats_per_cta(C.P, batch);
  M.long_scratch = {off, M.long_scratch_floats * sizeof(float) * PMT_PARTIAL_CTAS};
  off = align_to(off + M.long_scratch.bytes, 256);
  M.tile_slot = off;
  M.tiles = {0, tile_list_bytes(B)};
  M.perm = {M.tiles.bytes, perm_bytes(B)};
  M.claims = {0, C.saved.total > 0 ? pmt_plan_claim_bytes(B, PMT_PARTIAL_CTAS) : 0};
  off = align_to(off + std::max(M.perm.off + M.perm.bytes + 256, M.claims.bytes), 256);
  M.long_slot = off;
  off = align_to(off + (C.lng == LongKernel::TC ? C.long_tc.bytes + 1024 : 0), 256);
  M.cnn_tail = {off, cnn_tail_bytes(C, B)};
  M.end = off + M.cnn_tail.bytes + 1024;
  return M;
}

// Long-set kernel of the SIMT backward: every chunk of the longest set has its own recompute scratch + dL/dx + gate state
// (see the kernel).  The grid shrinks when the scratch of a full grid would pass kLongScratchBudget.
static const size_t kLongScratchBudget = (size_t)16 << 30;
static size_t long_bwd_floats_per_cta(const Plan& P, const PmtBatch* batch) {
  if (!batch || !pmt_has_long_sets(batch)) return 0;
  const size_t chunks = (size_t)((batch->max_rows_per_variant + 3 + TILE - 1) / TILE);
  return chunks * ((size_t)P.scratch_floats + (size_t)(P.d.d_model + 3 * P.d.d_ffn) * LD);
}
static int long_bwd_grid(const Plan& P, const PmtBatch* batch) {
  const size_t per_cta = long_bwd_floats_per_cta(P, batch) * sizeof(float);
  if (per_cta == 0) return 0;
  size_t grid = kLongScratchBudget / per_cta;
  if (grid > (size_t)PMT_PARTIAL_CTAS) grid = PMT_PARTIAL_CTAS;
  if (grid > (size_t)batch->n_variants) grid = batch->n_variants;
  return grid < 1 ? 1 : (int)grid;
}

static BwdMap backward_map(const CallPlan& C, const PmtBatch* batch) {
  const Plan& P = C.P;
  const size_t w = batch ? (size_t)batch->n_variants * (P.d.d_info + P.d.d_seq) * sizeof(float) : 0;
  BwdMap M;
  memset(&M, 0, sizeof(M));
  M.scr_floats = P.scratch_floats > P.info_scratch_floats ? P.scratch_floats : P.info_scratch_floats;
  M.long_grid = long_bwd_grid(P, batch);
  M.long_floats = long_bwd_floats_per_cta(P, batch);
  size_t off = 256;
  M.image = {off, pmt_image_bytes(P, C.G)};
  off = align_to(off + M.image.bytes, 256);
  M.partials = {off, (size_t)PMT_PARTIAL_CTAS * P.d.n_params * sizeof(float)};
  off += M.partials.bytes;
  M.scratch = {off, (size_t)PMT_PARTIAL_CTAS * M.scr_floats * sizeof(float)};
  off += M.scratch.bytes;
  M.info_seq = {off, w};
  off += w;
  M.d_info_seq = {off, w};
  off = align_to(off + w, 256);
  M.long_scratch = {off, (size_t)M.long_grid * M.long_floats * sizeof(float)};
  off = align_to(off + M.long_scratch.bytes, 256);
  M.tc_slot = off;
  off = align_to(off + (C.bwd_reads_tc ? C.tc_bwd.total + 1024 : 0), 256);
  M.cnn_slot = off;
  if (C.bwd_cnn_tc) {
    const int n = batch && batch->n_variants < PMT_CNN_BWD_CHUNK ? batch->n_variants : PMT_CNN_BWD_CHUNK;
    const size_t groups = ((size_t)n + C.C.G - 1) / C.C.G;
    M.cnn_fwd_image = {0, pmt_cnn_tc_image_bytes(C)};
    M.cnn_bwd_image = {align_to(M.cnn_fwd_image.bytes, 256), (size_t)C.CB.img_total * sizeof(float)};
    M.cnn_save = {M.cnn_bwd_image.off + align_to(M.cnn_bwd_image.bytes, 256), groups * C.CB.group_floats * sizeof(float)};
    off += M.cnn_fwd_image.bytes + 256 + M.cnn_bwd_image.bytes + 256 + M.cnn_save.bytes + 1024;
  }
  M.end = off;
  return M;
}

void pmt_plan_workspaces(CallPlan& C, const PmtBatch* batch) {
  C.fwd = forward_map(C, batch);
  C.bwd = backward_map(C, batch);
}

extern "C" size_t pmt_workspace_size(const PmtModelDesc* desc, const PmtBatch* batch, int for_backward) {
  CallPlan C;
  if (pmt_call_plan(desc, batch, false, &C)) return 0;
  return for_backward ? C.bwd.end : C.fwd.end;
}

extern "C" size_t pmt_train_saved_bytes(const PmtModelDesc* desc, const PmtBatch* batch) {
  CallPlan C;
  if (pmt_call_plan(desc, batch, true, &C)) return 0;
  return C.saved.total;
}

// ---- the resolvers ----

namespace {
// A caller's buffer [base, base + bytes); `fits` turns false once a resolved region ends past it.
struct Carve {
  unsigned char* base;
  size_t bytes;
  bool fits;
  // the offset of the first address at or after base + off that is a multiple of `align`
  size_t realign(size_t off, size_t align) const { return (size_t)(pmt_align_up(base + off, align) - base); }
  // region r of the slot at offset `slot`, realigned to `align`
  template <class T>
  T* at(const Region& r, size_t align = 1, size_t slot = 0) {
    const size_t off = realign(slot + r.off, align);
    if (off + r.bytes > bytes) fits = false;
    return reinterpret_cast<T*>(base + off);
  }
};
}  // namespace

int pmt_forward_buffers(const CallPlan& C, void* workspace, size_t bytes, FwdBuffers* out) {
  const FwdMap& M = C.fwd;
  PMT_CHECK(workspace && bytes >= M.end, "workspace too small: %zu < %zu", bytes, M.end);
  Carve K{reinterpret_cast<unsigned char*>(workspace), bytes, true};
  FwdBuffers W{};
  W.counters = K.at<int>(M.counters);
  W.image = K.at<float>(M.image);
  W.tc_image = K.at<unsigned char>(M.tc_image, 1024);
  W.cnn_tc_image = K.at<unsigned char>(M.cnn_tc_image);
  W.info_seq = K.at<float>(M.info_seq);
  W.long_scratch = K.at<float>(M.long_scratch);
  const size_t tile_slot = K.realign(M.tile_slot, 256);
  W.tiles = K.at<int>(M.tiles, 1, tile_slot);
  if (C.packed_planner) W.perm = K.at<int>(M.perm, 1, tile_slot);
  W.claims = K.at<int>(M.claims, 1, tile_slot);
  if (C.lng == LongKernel::TC) {
    const LongLayout& L = C.long_tc;
    const size_t long_slot = K.realign(M.long_slot, 256);
    W.lng.list = K.at<int>(L.list, 1, long_slot);
    W.lng.n_tiles = K.at<int>(L.n_tiles, 1, long_slot);
    W.lng.tiles = K.at<LongTile>(L.tiles, 1, long_slot);
    W.lng.counters = K.at<int>(L.counters, 1, long_slot);
    W.lng.fin_cnt = K.at<int>(L.fin_cnt, 1, long_slot);
    W.lng.mf_part = K.at<float>(L.mf_part, 1, long_slot);
    W.lng.fin_part = K.at<float>(L.fin_part, 1, long_slot);
  }
  W.cnn_tail = K.at<float>(M.cnn_tail);
  PMT_CHECK(K.fits, "forward workspace map: a region ends past the %zu-byte buffer", bytes);
  *out = W;
  return 0;
}

int pmt_backward_buffers(const CallPlan& C, void* workspace, size_t bytes, BwdBuffers* out) {
  const BwdMap& M = C.bwd;
  PMT_CHECK(workspace && bytes >= M.end, "workspace too small: %zu < %zu", bytes, M.end);
  Carve K{reinterpret_cast<unsigned char*>(workspace), bytes, true};
  BwdBuffers W{};
  W.image = K.at<float>(M.image);
  W.partials = K.at<float>(M.partials);
  W.scratch = K.at<float>(M.scratch);
  W.info_seq = K.at<float>(M.info_seq);
  W.d_info_seq = K.at<float>(M.d_info_seq);
  W.long_scratch = K.at<float>(M.long_scratch);
  if (C.bwd_reads_tc) {
    const BwdLayout& L = C.tc_bwd;
    const size_t tc = K.realign(M.tc_slot, 1024);
    W.tc.image_f = K.at<unsigned char>(L.image_f, 1, tc);
    W.tc.image_t = K.at<unsigned char>(L.image_t, 1, tc);
    W.tc.tiles = K.at<int>(L.tiles, 1, tc);
    W.tc.claims = K.at<int>(L.claims, 1, tc);
    W.tc.partials = K.at<float>(L.partials, 1, tc);
    W.tc.reduced = K.at<float>(L.reduced, 1, tc);
    W.tc.scratch = K.at<unsigned char>(L.scratch, 1, tc);
  }
  if (C.bwd_cnn_tc) {
    const size_t cnn = K.realign(M.cnn_slot, 256);
    W.cnn.fwd_image = K.at<unsigned char>(M.cnn_fwd_image, 1, cnn);
    W.cnn.bwd_image = K.at<float>(M.cnn_bwd_image, 1, cnn);
    W.cnn.save = K.at<float>(M.cnn_save, 1, cnn);
  }
  PMT_CHECK(K.fits, "backward workspace map: a region ends past the %zu-byte buffer", bytes);
  *out = W;
  return 0;
}

int pmt_saved_buffers(const CallPlan& C, const void* saved, size_t bytes, SavedBuffers* out) {
  const SavedLayout& S = C.saved;
  PMT_CHECK(saved && S.total > 0 && bytes >= S.total, "saved buffer too small: %zu < %zu", bytes, S.total);
  Carve K{const_cast<unsigned char*>(reinterpret_cast<const unsigned char*>(saved)), bytes, true};
  SavedBuffers W{};
  W.tiles = K.at<int>(S.tiles);
  W.scratch = K.at<unsigned char>(S.scratch);
  W.cnn = K.at<float>(S.cnn);
  PMT_CHECK(K.fits, "saved-buffer map: a region ends past the %zu-byte buffer", bytes);
  *out = W;
  return 0;
}
