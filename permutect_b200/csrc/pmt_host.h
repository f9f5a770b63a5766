// Host-side helpers shared by the translation units of libpermutect_b200.so.
#pragma once
#include <cstdarg>
#include <cstddef>

#include "pmt_device.cuh"

void pmt_set_error(const char* fmt, ...);
#define PMT_CHECK(cond, ...)     \
  do {                           \
    if (!(cond)) {               \
      pmt_set_error(__VA_ARGS__); \
      return 1;                  \
    }                            \
  } while (0)

// CUDA runtime calls whose failure would otherwise only surface as a later launch error (opt-in shared memory, memsets)
#define PMT_CUDA(call)                                                                        \
  do {                                                                                        \
    cudaError_t pmt_cuda_err_ = (call);                                                       \
    if (pmt_cuda_err_ != cudaSuccess) {                                                       \
      pmt_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(pmt_cuda_err_), __FILE__, __LINE__); \
      return 1;                                                                               \
    }                                                                                         \
  } while (0)

// The first address at or after `p` that is a multiple of `align` (a power of two): the C-ABI does not require aligned
// buffers, so regions that a kernel needs aligned are realigned inside the caller's buffer.
inline unsigned char* pmt_align_up(void* p, size_t align) {
  return reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(p) + align - 1) & ~(uintptr_t)(align - 1));
}

// A set occupies pad4(ref rows) + alt rows of a tile, so a set of up to TILE - 3 rows always fits in one tile; anything
// longer MAY be left to the long-set kernels by build_tile / plan_tiles_kernel (which then do nothing if it did fit).
inline bool pmt_has_long_sets(const PmtBatch* batch) { return batch->max_rows_per_variant + 3 > PMT_TILE_ROWS; }

int pmt_build_plan(const PmtModelDesc* d, pmt::Plan* out);
int pmt_cnn_geometry(const pmt::Plan& P, pmt::CnnGeom* out);
size_t pmt_image_bytes(const pmt::Plan& P, const pmt::CnnGeom& G);
void pmt_profile_begin(cudaStream_t st);
void pmt_profile_end(cudaStream_t st);
int pmt_precision_mode();
int pmt_posterior_ctas_override();
