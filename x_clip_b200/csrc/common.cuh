// Device-side primitives for the sm_100a kernels of x_clip_b200: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (UMMA + TMEM) and descriptor builders.
//
// Everything here is inline PTX; nothing depends on CUTLASS/CuTe.  Bit layouts of
// the shared-memory matrix descriptor and the instruction descriptor follow the
// PTX ISA "tcgen05" chapter (the same fields CuTe names in
// cute/arch/mma_sm100_desc.hpp: start_address[0,14) LBO[16,30) SBO[32,46)
// version[46,48) layout_type[61,64); idesc: c_format[4,6) a_format[7,10)
// b_format[10,13) a_major[15] b_major[16] n>>3[17,23) m>>4[24,29)).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>
#include <stdio.h>

namespace xclip {

typedef __nv_bfloat16 bf16;

constexpr int kMajorK = 0;   // operand stored with the contraction index contiguous
constexpr int kMajorMN = 1;  // operand stored with its M (or N) index contiguous

// ---------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

// Single-thread regions that issue tcgen05.mma / TMA instructions are entered through
// elect.sync: with `lane == 0` ptxas cannot prove that one thread is active, so every UTCHMMA /
// UTMALDG got a waterfall loop (ELECT + BRA.U.ANY + R2UR, ~17 SASS instructions per MMA instead
// of ~8).  Validated on a B200 in round 2 (full GPU suite; attention backward 1.91 -> 1.80 ms).
#define XCLIP_ONE_LANE(lane) (::xclip::elect_one())

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}

// ---------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)
               : "memory");
}

__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// make generic-proxy writes to shared memory visible to the async proxy (TMA, UMMA)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}

// Bounded wait: a protocol bug turns into a trap (launch failure the host reports)
// instead of a hung GPU.  ~4 s at 2 GHz.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 8000000000ll) {
      printf("xclip: mbarrier timeout block=(%d,%d) thread=%d bar=%u parity=%u\n", blockIdx.x,
             blockIdx.y, threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ---------------------------------------------------------------------------
// CTA pair (cta_group::2) primitives: two CTAs of a 2-cluster issue ONE tcgen05.mma of M = 256;
// each CTA stages its own 128 rows of A and its own half of B's N columns, so the operand bytes
// every SM pulls from L2 per flop drop by a third against two independent 128 x 256 tiles.
// PTX forms as in CUTLASS (cute/arch/copy_sm100_tma.hpp, mma_sm100_umma.hpp, cutlass/arch/barrier.h).
// ---------------------------------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are credited to the mbarrier of the pair's LEADER (even) CTA
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                                 int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair_512(uint32_t* smem_result) {  // whole warp, BOTH CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(512)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair_512(uint32_t taddr) {  // whole warp, BOTH CTAs
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(512) : "memory");
}
// D[tmem of both CTAs, M = 256] (+)= A * B; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at the same smem offset in BOTH CTAs once all prior MMAs retired
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(static_cast<uint16_t>(3))
      : "memory");
}
// plain arrive on the LEADER CTA's copy of a barrier (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask)
               : "memory");
}

// ---------------------------------------------------------------------------
// tcgen05: TMEM allocation, MMA, commit, loads, fences
// ---------------------------------------------------------------------------
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {  // whole warp
  static_assert(kCols == 32 || kCols == 64 || kCols == 128 || kCols == 256 || kCols == 512, "");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}

template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
               : "memory");
}

__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// mbarrier arrive when all previously issued tcgen05.mma of this thread completed.
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives lane
// (lane_base + t), columns [col, col+32).  A warp may only touch the lane quarter
// 32*(warp_id%4)..+31.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
        "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------------
// descriptors
// ---------------------------------------------------------------------------
// Shared-memory matrix descriptor for a SWIZZLE_128B tile whose base is 1024 B aligned.
//   K-major  : rows (M/N index) of 128 B (64 bf16 along K); 8-row groups SBO apart
//              (1024 B when the tile is dense); LBO unused.
//   MN-major : rows (K index) of 128 B (64 bf16 along M/N); 8-row K-groups SBO apart
//              (1024 B); 64-element M/N groups LBO apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;  // SWIZZLE_128B
  return d;
}

// advance a descriptor's start address by `bytes` (must keep the 1024 B swizzle phase)
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) {
  return desc + static_cast<uint64_t>(bytes >> 4);
}

// kind::f16 instruction descriptor: bf16 x bf16 -> fp32
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_major, int b_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_major) << 15) |
         (static_cast<uint32_t>(b_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// byte offset of 16 B chunk `c16` of 128 B row `row` inside a SWIZZLE_128B tile
// (Swizzle<3,4,3>: chunk index XOR row%8); tile base must be 1024 B aligned.
__device__ __forceinline__ uint32_t swz128(uint32_t row, uint32_t c16) {
  return row * 128u + ((c16 ^ (row & 7u)) << 4);
}

// ---------------------------------------------------------------------------
// Packed fp32x2 arithmetic (sm_100: FFMA2 - one instruction, one issue slot, two IEEE fp32 FMAs on
// an aligned register pair).  The GELU epilogues of the fused feed-forward are bound by the FMA pipe
// (~28 FMA-class instructions per element in scalar form against 2 MUFU); in packed form the
// polynomial and the affine chains cost half the instructions and the two MUFU become the floor.
// ---------------------------------------------------------------------------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 f2_pack(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ f32x2 f2_splat(float v) { return f2_pack(v, v); }
__device__ __forceinline__ void f2_unpack(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 f2_mul(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 f2_add(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// two consecutive bf16 of one 32-bit word -> packed fp32 pair (element 0 in the low half)
__device__ __forceinline__ f32x2 f2_from_bf16x2(uint32_t w) {
  return f2_pack(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ uint32_t f2_to_bf16x2(f32x2 v) {
  float lo, hi;
  f2_unpack(v, lo, hi);
  return pack_bf16x2(lo, hi);
}

// ---------------------------------------------------------------------------
// GELU (erf form, x_clip/x_clip.py:183 F.gelu) for the fused feed-forward GEMM epilogues, two elements
// at once: cdf = Phi(x) = 0.5 * (1 + erf(x / sqrt(2))), pdf = phi(x) = exp(-x^2/2) / sqrt(2 pi).
// erf by Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7, far below bf16 output resolution): one
// MUFU.RCP + one MUFU.EX2 + 6 FMA per element instead of libdevice erff's ~25 instructions.
// exp(-x^2/2) is shared with the Gaussian density that gelu'(x) needs.
// ---------------------------------------------------------------------------
struct GeluParts2 {
  f32x2 cdf, pdf;
};
__device__ __forceinline__ GeluParts2 gelu_parts2(float x0, float x1) {
  const f32x2 x = f2_pack(x0, x1);
  const f32x2 z = f2_mul(f2_pack(fabsf(x0), fabsf(x1)), f2_splat(0.70710678118654752f));
  float d0, d1, t0, t1;
  f2_unpack(f2_fma(f2_splat(0.3275911f), z, f2_splat(1.f)), d0, d1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
  const f32x2 t = f2_pack(t0, t1);
  f32x2 poly = f2_fma(f2_splat(1.061405429f), t, f2_splat(-1.453152027f));
  poly = f2_fma(poly, t, f2_splat(1.421413741f));
  poly = f2_fma(poly, t, f2_splat(-0.284496736f));
  poly = f2_fma(poly, t, f2_splat(0.254829592f));
  poly = f2_mul(poly, t);
  float a0, a1, e0, e1;
  f2_unpack(f2_mul(f2_mul(x, f2_splat(-0.72134752044448170f)), x), a0, a1);     // -x^2/2 * log2(e)
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(a0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(a1));
  const f32x2 e_half = f2_pack(e0, e1);
  // q = 0.5 - 0.5 erfc(|x|/sqrt2) >= 0;  Phi(x) = 0.5 + sign(x) q
  float q0, q1;
  f2_unpack(f2_fma(f2_mul(poly, e_half), f2_splat(-0.5f), f2_splat(0.5f)), q0, q1);
  q0 = __uint_as_float(__float_as_uint(q0) | (__float_as_uint(x0) & 0x80000000u));
  q1 = __uint_as_float(__float_as_uint(q1) | (__float_as_uint(x1) & 0x80000000u));
  GeluParts2 g;
  g.cdf = f2_add(f2_pack(q0, q1), f2_splat(0.5f));
  g.pdf = f2_mul(e_half, f2_splat(0.3989422804014327f));
  return g;
}


}  // namespace xclip
