// PTX wrappers for the tcgen05 / TMEM / mbarrier / fence / bulk-copy instructions used by the tensor-core kernels, and the
// shared-memory descriptors of their MMA operands (sm_100a).
#pragma once
#include <cstdint>

#include "pmt_device.cuh"

namespace pmt {
namespace tc {

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (tcgen05.mma operands, bulk copies)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: the warp sleeps in hardware until the phase completes (or the hint expires) instead
// of polling -- a polling loop takes issue slots from the epilogue warps that share the SM sub-partition.
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(0x989680u)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void slot_barrier(int slot) { asm volatile("bar.sync %0, 128;" ::"r"(slot + 1) : "memory"); }
__device__ __forceinline__ bool elect_one() {
  unsigned pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// TMEM allocation of COLS columns for the CTA, written to shared memory at `slot`; called by one whole warp, which also
// deallocates.  Alloc and dealloc must name the same COLS.
template <int COLS>
__device__ __forceinline__ void tmem_alloc(unsigned slot) {
  static_assert(COLS >= 32 && COLS <= 512 && (COLS & (COLS - 1)) == 0, "TMEM allocations are a power of two, 32 to 512 columns");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(COLS));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(unsigned base) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(COLS));
}

// ---------------------------------------------------------------- shared-memory descriptors
__device__ __forceinline__ uint64_t smem_desc(unsigned addr) {
  // K-major, SWIZZLE_128B: 8-row groups 1024 B apart, descriptor version 1 (sm_100)
  return (uint64_t)((addr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// K-major, no swizzle.  Low word: start address >> 4 | (LBO >> 4) << 16 with LBO = the distance between K-adjacent core
// matrices; high word (constant): SBO = 128 B between 8-row groups, descriptor version 1.
constexpr unsigned DESC_HI = 8u | (1u << 14);
__device__ __forceinline__ unsigned desc_lo(unsigned addr, unsigned lbo_bytes) { return ((addr >> 4) & 0x3FFFu) | ((lbo_bytes >> 4) << 16); }
// MN-major tf32 operand made of panels, SWIZZLE_128B_BASE32B: MN atoms (32 features) panel_bytes apart, K atoms (4 rows)
// 512 bytes apart (profiles/microbench/wgrad_probe.cu)
__device__ __forceinline__ uint64_t desc_panels(unsigned addr, unsigned panel_bytes) {
  return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)(panel_bytes >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (1ull << 61);
}
// Instruction descriptor of kind::tf32, M = 128, N columns: fp32 accumulator, both operands K-major
__host__ __device__ constexpr unsigned make_idesc(int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(N >> 3) << 17) | ((128u >> 4) << 24);
}

// ---------------------------------------------------------------- MMAs (kind::tf32, accumulate into TMEM unless accumulate == 0)
// A and B in shared memory, given by the low words of no-swizzle descriptors (desc_lo; high word DESC_HI)
template <unsigned IDESC>
__device__ __forceinline__ void mma_ss_desc_lo(unsigned tmem_d, unsigned a_lo32, unsigned b_lo32, unsigned accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %3, 0;\n\t"
      "mov.b64 da, {%1, %4};\n\t"
      "mov.b64 db, {%2, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}" ::"r"(tmem_d),
      "r"(a_lo32), "r"(b_lo32), "r"(accumulate), "n"(DESC_HI), "n"(IDESC)
      : "memory");
}
// A and B in shared memory, given by full 64-bit descriptors
__device__ __forceinline__ void mma_ss_desc64(unsigned tmem_d, uint64_t adesc, uint64_t bdesc, unsigned idesc, unsigned accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A in TMEM, B in shared memory (64-bit descriptor)
__device__ __forceinline__ void mma_ts(unsigned tmem_d, unsigned tmem_a, uint64_t bdesc, unsigned idesc, unsigned accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_commit(unsigned bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

#define PMT_R8(r, o) "=r"(r[o]), "=r"(r[o + 1]), "=r"(r[o + 2]), "=r"(r[o + 3]), "=r"(r[o + 4]), "=r"(r[o + 5]), "=r"(r[o + 6]), "=r"(r[o + 7])
#define PMT_W8(r, o) "r"(r[o]), "r"(r[o + 1]), "r"(r[o + 2]), "r"(r[o + 3]), "r"(r[o + 4]), "r"(r[o + 5]), "r"(r[o + 6]), "r"(r[o + 7])

// 32 lanes x 32 bit: thread t of the warp gets columns [col, col + n) of its TMEM lane
__device__ __forceinline__ void tmem_ld8(unsigned taddr, unsigned* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : PMT_R8(r, 0) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(unsigned taddr, unsigned* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : PMT_R8(r, 0), PMT_R8(r, 8)
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32(unsigned taddr, unsigned* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,"
      "%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : PMT_R8(r, 0), PMT_R8(r, 8), PMT_R8(r, 16), PMT_R8(r, 24)
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st4(unsigned taddr, const unsigned* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%4], {%0,%1,%2,%3};" ::"r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st8(unsigned taddr, const unsigned* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%8], {%0,%1,%2,%3,%4,%5,%6,%7};" ::PMT_W8(r, 0), "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st16(unsigned taddr, const unsigned* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%16], {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15};" ::PMT_W8(r, 0),
               PMT_W8(r, 8), "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st32(unsigned taddr, const unsigned* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,"
      "%23,%24,%25,%26,%27,%28,%29,%30,%31};" ::PMT_W8(r, 0),
      PMT_W8(r, 8), PMT_W8(r, 16), PMT_W8(r, 24), "r"(taddr)
      : "memory");
}

// Paired FP32 (FFMA2 / FADD2 / FMUL2): two independent lanes, each rounded exactly as the scalar instruction would round it
// (round-to-nearest, no flush to zero), so pairing changes no value.  nvcc does not pair scalar code on its own.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void up2(f32x2 r, float& a, float& b) { asm("mov.b64 {%0,%1}, %2;" : "=f"(a), "=f"(b) : "l"(r)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) { f32x2 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// u(x) = x > 0 ? x : alpha (e^x - 1); selu(x) = scale * u(x).  The scale is folded into the consuming weights
// wherever a SELU output feeds a Linear layer.
__device__ __forceinline__ float selu_u(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 1.4426950408889634f));
  const float neg = fmaf(SELU_ALPHA, e, -SELU_ALPHA);
  return x > 0.f ? x : neg;
}
// selu_u of v[0..N), bitwise equal to N selu_u calls: the exponent arguments are paired multiplies.  The alpha FMA stays
// scalar: it is predicated on x <= 0, which a paired FMA would turn into an FMA plus a select.
template <int N>
__device__ __forceinline__ void selu_u_n(float* v) {
  static_assert(N % 2 == 0, "pairs");
  const f32x2 l2e = pk2(1.4426950408889634f, 1.4426950408889634f);
#pragma unroll
  for (int i = 0; i < N; i += 2) {
    float t0, t1, e0, e1;
    up2(mul2(pk2(v[i], v[i + 1]), l2e), t0, t1);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(t0));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(t1));
    v[i] = v[i] > 0.f ? v[i] : fmaf(SELU_ALPHA, e0, -SELU_ALPHA);
    v[i + 1] = v[i + 1] > 0.f ? v[i + 1] : fmaf(SELU_ALPHA, e1, -SELU_ALPHA);
  }
}

__device__ __forceinline__ float lds_f32(unsigned a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_f32(unsigned a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ float2 lds_f32x2(unsigned a) { float2 v; asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ void sts_f32x2(unsigned a, float x, float y) { asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(a), "f"(x), "f"(y) : "memory"); }
__device__ __forceinline__ int lds_s32(unsigned a) { int v; asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ long long lds_s64(unsigned a) { long long v; asm volatile("ld.shared.s64 %0, [%1];" : "=l"(v) : "r"(a)); return v; }
__device__ __forceinline__ unsigned lds_u8(unsigned a) { unsigned v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void named_barrier(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }


}  // namespace tc
}  // namespace pmt
