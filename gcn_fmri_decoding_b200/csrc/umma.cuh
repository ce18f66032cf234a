// Blackwell (sm_100a) primitives of the tcgen05 kernels: mbarriers, TMEM allocation, shared-memory matrix
// descriptors, tcgen05.mma / commit / ld, and the shared-memory layouts the kernels keep their operands in.
//
// Operand layouts (all K-major, i.e. the contraction index runs fastest inside a row):
//   state slab   fp32 [rows][32]  128-byte rows, 8-row atoms of 1 KB, SWIZZLE_128B: the 16-byte chunk c of row r sits
//                at chunk position c ^ (r & 7).  One row = G windows x FP features (G*FP = 32).  The SIMT sparse
//                step gathers whole rows (8 lanes x 16 B = one conflict-free wavefront) and tcgen05.mma reads the
//                very same bytes as its A operand (kind::tf32 ignores the low 13 mantissa bits = the "hi" part).
//   lo slab      bf16 [rows][32]  64-byte rows, 8-row atoms of 512 B, SWIZZLE_64B: chunk c ^ ((r >> 1) & 3).  Holds
//                x - trunc_tf32(x), the error-compensation term of the split product (kind::f16, bf16 inputs).
//   taps         [N = 32 filters][Ktot] no swizzle: core matrices of 8 filters x 16 bytes, core (kc, ng) at
//                ((kc * 4) + ng) * 128 bytes (LBO = 512 B between K chunks, SBO = 128 B between filter groups).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace gcnb {
namespace um {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier -----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch failure (trap), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}

// Long waits (a whole tile): poll every ~100 ns instead of spinning -- the pollers share their schedulers with the one
// thread that issues the MMAs, and every issue slot they burn delays it.
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(100);
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}

// TMA bulk copy global -> shared (16-byte aligned addresses, size a multiple of 16), completion on an mbarrier
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  __syncwarp();  // bar.sync is an aligned barrier: the warp must arrive converged (lanes may have left a loop separately)
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// one lane of the (converged) warp; ptxas knows a single thread is active under this predicate
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ---- TMEM ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- descriptors --------------------------------------------------------------------------------------------
// 64-bit shared-memory matrix descriptor: start address, leading / stride byte offsets (16-byte units),
// version 1 (Blackwell), swizzle mode in bits 61..63.
enum : uint64_t { kSwzNone = 0, kSwz128 = 2, kSwz64 = 4, kSwz32 = 6 };
__host__ __device__ constexpr uint64_t smem_desc_base(uint32_t lbo_bytes, uint32_t sbo_bytes, uint64_t swizzle) {
  return ((uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32) | (1ull << 46) |
         (swizzle << 61);
}
__device__ __forceinline__ uint64_t smem_desc(uint64_t base, uint32_t addr) { return base | ((addr >> 4) & 0x3fff); }

constexpr uint64_t kDescSlab = smem_desc_base(16, 1024, kSwz128);  // fp32 state rows (A operand, tf32 passes)
constexpr uint64_t kDescLo = smem_desc_base(16, 512, kSwz64);      // bf16 compensation rows (A operand, bf16 pass)
constexpr uint64_t kDescTaps = smem_desc_base(512, 128, kSwzNone); // taps (B operand), N = 32

// 32-bit instruction descriptor: D fp32, A/B format (0 f16, 1 bf16, 2 tf32), both K-major, N >> 3, M >> 4.
__host__ __device__ constexpr uint32_t instr_desc(uint32_t ab_format, uint32_t M, uint32_t N) {
  return (1u << 4) | (ab_format << 7) | (ab_format << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
constexpr uint32_t kIdescTf32 = instr_desc(2, 128, 32);
constexpr uint32_t kIdescBf16 = instr_desc(1, 128, 32);
// N = 16: the same tap layout, only its first two 8-filter groups are read (outputs of at most 16 columns)
constexpr uint32_t kIdescTf32N16 = instr_desc(2, 128, 16);
constexpr uint32_t kIdescBf16N16 = instr_desc(1, 128, 16);

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread on behalf of the CTA.
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once every tcgen05.mma this thread issued so far has completed (implies fence::before).
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives row (lane base + t), columns col..col+31.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- shared-memory access by 32-bit shared address ------------------------------------------------------------
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ int4 lds128i(uint32_t a) {
  int4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint2 lds64u(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds32u(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}

// ---- packed fp32 pairs (fma.rn.f32x2: two independent IEEE fp32 FMAs in one issue slot) ------------------------------
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// ---- operand layouts ----------------------------------------------------------------------------------------
// byte offset of 16-byte chunk c (0..7) of state row r inside a slab
__device__ __forceinline__ uint32_t slab_off(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }
// gather code of a neighbour row: XOR with (c << 4) gives slab_off(col, c)
__host__ __device__ __forceinline__ uint32_t gather_code(int col) { return (uint32_t)((col << 7) | ((col & 7) << 4)); }
// byte offset of the 8-byte half-chunk holding features 4c..4c+3 (bf16) of lo row r
__device__ __forceinline__ uint32_t lo_off(int r, int c) {
  return (uint32_t)(r * 64 + ((((c >> 1) ^ ((r >> 1) & 3)) << 4) | ((c & 1) << 3)));
}
// byte offsets of tap element (kk = contraction index, o = filter) in the tf32 / bf16 tap images (N = 32)
__host__ __device__ __forceinline__ uint32_t tap_off_tf32(int kk, int o) {
  return (uint32_t)((((kk >> 2) * 4 + (o >> 3)) * 128) + (o & 7) * 16 + (kk & 3) * 4);
}
__host__ __device__ __forceinline__ uint32_t tap_off_bf16(int kk, int o) {
  return (uint32_t)((((kk >> 3) * 4 + (o >> 3)) * 128) + (o & 7) * 16 + (kk & 7) * 2);
}

__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
// what kind::tf32 sees of an fp32 operand: the low 13 mantissa bits are dropped
__device__ __forceinline__ float tf32_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// Store four consecutive features of one state row: the fp32 value into the slab and its tf32 remainder (bf16)
// into the lo slab.
__device__ __forceinline__ void store_state(uint32_t slab, uint32_t lo, int row, int c, float4 v) {
  sts128(slab + slab_off(row, c), v);
  const float rx = v.x - tf32_trunc(v.x), ry = v.y - tf32_trunc(v.y);
  const float rz = v.z - tf32_trunc(v.z), rw = v.w - tf32_trunc(v.w);
  sts64(lo + lo_off(row, c), pack_bf16(rx, ry), pack_bf16(rz, rw));
}

// the same with both byte addresses already resolved
__device__ __forceinline__ void store_state_at(uint32_t slab_addr, uint32_t lo_addr, float4 v) {
  sts128(slab_addr, v);
  const float rx = v.x - tf32_trunc(v.x), ry = v.y - tf32_trunc(v.y);
  const float rz = v.z - tf32_trunc(v.z), rw = v.w - tf32_trunc(v.w);
  sts64(lo_addr, pack_bf16(rx, ry), pack_bf16(rz, rw));
}

}  // namespace um
}  // namespace gcnb
