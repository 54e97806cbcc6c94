// Thin inline-PTX wrappers for the sm_100a features the kernels use: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (alloc / mma / commit / ld) and the UMMA shared-memory + instruction descriptors.
// Written from the PTX ISA; no CUTLASS/CuTe dependency.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace wj {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, 0xFFFFFFFF;\n"
      "selp.u32 %0, 1, 0, px;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// Wait for roles that are usually far ahead of the barrier (the TMA producer on a full ring, the MMA warp on an
// accumulator the epilogue still reads): after a failed probe the warp sleeps instead of re-issuing the probe every
// ~16 cycles, which would take issue slots from the epilogue warps of the same scheduler.
template <int NS = 64>
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  uint32_t addr = static_cast<uint32_t>(__cvta_generic_to_shared(bar));
  uint32_t ok;
  for (;;) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) break;
    __nanosleep(NS);
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  uint32_t ok;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// ----------------------------------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
      "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}

// L2 prefetch of a 2-D tile (no shared-memory destination, no barrier): the later tma_load_2d of the same box hits L2
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* tm, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1)
               : "memory");
}

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4),
      "r"(smem_u32(bar))
      : "memory");
}

// TMA store (smem -> global, bulk-group completion); rows / columns outside the tensor map are clipped by the hardware.
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------- tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], tf32 inputs (fp32 words whose low 13 mantissa bits the tensor core ignores), fp32
// accumulate, issued by ONE thread.  One instruction consumes 32 bytes of K (K = 8), like kind::f16 with K = 16.
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on `bar` once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i of the warp = TMEM lane base+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 16 TMEM lanes x 32 fp32 columns -> 16 registers per thread, mma-accumulator-like distribution: with g = lane / 4 and
// tg = lane % 4, v[4*j + 2*hr + e] = (TMEM lane base + g + 8*hr, column 8*j + 2*tg + e), j = 0..3, hr, e = 0..1.
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
// 4x4 transpose of 64-bit items across a quad of lanes (tg = lane % 4): in: a[2j], a[2j+1] = item j of this lane;
// out: a[2j], a[2j+1] = item tg of lane j.  Two xor-shuffle rounds, 8 SHFL.
__device__ __forceinline__ void quad_exchange(uint32_t& lo0, uint32_t& lo1, uint32_t& hi0, uint32_t& hi1, bool has_bit,
                                              int bit) {
  const uint32_t x0 = has_bit ? lo0 : hi0, x1 = has_bit ? lo1 : hi1;
  const uint32_t y0 = __shfl_xor_sync(0xffffffffu, x0, bit), y1 = __shfl_xor_sync(0xffffffffu, x1, bit);
  if (has_bit) { lo0 = y0; lo1 = y1; } else { hi0 = y0; hi1 = y1; }
}
__device__ __forceinline__ void quad_transpose(uint32_t (&a)[8], int tg) {
  quad_exchange(a[0], a[1], a[2], a[3], (tg & 1) != 0, 1);
  quad_exchange(a[4], a[5], a[6], a[7], (tg & 1) != 0, 1);
  quad_exchange(a[0], a[1], a[4], a[5], (tg & 2) != 0, 2);
  quad_exchange(a[2], a[3], a[6], a[7], (tg & 2) != 0, 2);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor (PTX ISA "tcgen05 shared memory descriptor"):
//   [0,14) start address >> 4, [16,30) leading byte offset >> 4, [32,46) stride byte offset >> 4,
//   [46,48) version = 1, [61,64) swizzle mode (2 = 128-byte).
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16 with bf16 A/B and fp32 D.
//   [4,6) D format (1 = f32), [7,10) A format (1 = bf16), [10,13) B format, bit 15 A major (1 = MN), bit 16 B major,
//   [17,23) N >> 3, [24,29) M >> 4.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
         (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}
// Instruction descriptor for kind::tf32 with tf32 A/B (format 2 in both fields), fp32 D, both operands K-major.
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// ----------------------------------------------------------------------------------------------- CTA pair (cta_group::2)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_smem_addr` in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads issued by either CTA of a pair: data lands in the issuing CTA's smem, the bytes are counted on the
// mbarrier `bar_cluster_addr` (the leader's barrier, a shared::cluster address).
__device__ __forceinline__ void tma_load_4d_pair(void* smem_dst, const CUtensorMap* tm, uint32_t bar_cluster_addr, int c0,
                                                 int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
      "r"(bar_cluster_addr)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tm, uint32_t bar_cluster_addr, int c0,
                                                 int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(bar_cluster_addr)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair(void* smem_dst, const CUtensorMap* tm, uint32_t bar_cluster_addr, int c0,
                                                 int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(bar_cluster_addr)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_pair(void* smem_dst, const CUtensorMap* tm, uint32_t bar_cluster_addr, int c0,
                                                 int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4),
      "r"(bar_cluster_addr)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot_in_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[256 x 16: 128 rows from each CTA's smem] * B[N x 16: N/2 rows from each CTA's smem],
// issued by ONE thread of the leader CTA.
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on the mbarrier at the same smem offset in BOTH CTAs once all previously issued pair MMAs have completed.
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "{\n"
      ".reg .b16 m;\n"
      "mov.b16 m, 3;\n"
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n"
      "}\n" ::"r"(smem_u32(bar))
      : "memory");
}

// Warpgroup register re-allocation (executed by all 4 warps of an aligned warpgroup).
template <int N>
__device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// ----------------------------------------------------------------------------------------------- misc math
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}
// erf-form GELU (approximate='none') without erff(): erfc(|x|/sqrt2) = poly(t) * exp(-x^2/2), t = 1/(1 + p|x|/sqrt2)
// (Abramowitz & Stegun 7.1.25, |error| <= 2.5e-5; every consumer rounds the result to bf16, eps 3.9e-3), so
//   gelu(x)  = max(x, 0) - 0.5 |x| erfc(|x|/sqrt2)            (no cancellation in the negative tail)
//   gelu'(x) = Phi(x) + x phi(x),  Phi = x > 0 ? 1 - 0.5 erfc : 0.5 erfc,  phi = exp(-x^2/2) / sqrt(2 pi)
// ~12 FMA-pipe + 2 MUFU instructions per value (|error| < 4e-7 for both on [-8, 8], checked against scipy).
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void gelu_terms(float x, float& ax, float& e, float& pe) {
  ax = fabsf(x);
  // erfc(z) = (a1 t + a2 t^2 + a3 t^3) exp(-z^2), t = 1 / (1 + p z), z = |x| / sqrt(2): Abramowitz & Stegun 7.1.25,
  // |error| <= 2.5e-5 -- two orders of magnitude below the bf16 rounding (2^-9) every result of these epilogues gets
  const float t = rcp_approx(fmaf(0.47047f * 0.70710678f, ax, 1.0f));
  float q = fmaf(t, 0.7478556f, -0.0958798f);
  q = fmaf(t, q, 0.3480242f);
  e = ex2_approx(-0.72134752f * x * x);
  pe = q * t * e;
}
__device__ __forceinline__ float gelu_fast(float x) {
  float ax, e, pe;
  gelu_terms(x, ax, e, pe);
  return fmaf(-0.5f * ax, pe, fmaxf(x, 0.0f));
}
__device__ __forceinline__ void gelu_fast2(float x, float& g, float& dg) {
  float ax, e, pe;
  gelu_terms(x, ax, e, pe);
  const float hp = 0.5f * pe;
  g = fmaf(-ax, hp, fmaxf(x, 0.0f));
  dg = fmaf(x * 0.39894228f, e, x > 0.0f ? 1.0f - hp : hp);
}
__device__ __forceinline__ float gelu_fast_grad(float x) {
  float g, dg;
  gelu_fast2(x, g, dg);
  return dg;
}
// ----------------------------------------------------------------------------------------------- packed-half GELU
// The GELU epilogues of the K = 384 GEMMs are ISSUE-bound (ncu: 72-77 % issue-slot utilisation with the tensor pipe at
// 36-54 %): a 128 x 256 tile with 6 k-blocks leaves ~12 issued instructions per output element, the fp32 erfc form
// above costs ~26 with the saved derivative.  Here two values share every instruction (HFMA2 / HMUL2 and ONE
// MUFU.TANH per pair):
//   Phi(x) ~= 0.5 (1 + tanh(x (C1 + C3 x^2))),  C1, C3 least-squares fitted to the erf form on [-6, 6]
//             (max |error| of Phi 1.6e-4; the textbook tanh-GELU constants give 1.8e-4)
//   gelu(x) = x Phi(x),  gelu'(x) = Phi(x) + 0.5 x (1 - t^2)(C1 + 3 C3 x^2)
// fp16 carries 3 more mantissa bits than the bf16 every result is rounded to, and the pre-activation enters as fp16
// instead of autocast's bf16, so against the fp32 reference the result is closer than the autocast-faithful fp32 path
// (rel-L2 of gelu 1.7e-3 vs 2.6e-3, gelu' 2.0e-3 vs 2.0e-3 on N(0,1) inputs; scripts/check_gelu_h2.py).
// Range: the conversion saturates at +-65504 and x^2 is clamped so that no inf * 0 can appear.
__device__ __forceinline__ __half2 h2_from_bits(uint32_t v) { return *reinterpret_cast<__half2*>(&v); }
__device__ __forceinline__ uint32_t h2_bits(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ __half2 h2_tanh_approx(__half2 x) {
  uint32_t y;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(y) : "r"(h2_bits(x)));
  return h2_from_bits(y);
}
__device__ __forceinline__ __half2 h2_pack_sat(float lo, float hi) {
  uint32_t y;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(y) : "f"(hi), "f"(lo));
  return h2_from_bits(y);
}
__device__ __forceinline__ uint32_t h2_to_bf16x2(__half2 v) {
  const float2 f = __half22float2(v);
  __nv_bfloat162 b = __floats2bfloat162_rn(f.x, f.y);
  return *reinterpret_cast<uint32_t*>(&b);
}
#define WJ_GELU_C1 0.79855342f
#define WJ_GELU_C3 0.03546201f
// (lo, hi) pre-activations -> packed bf16x2 gelu [and gelu']
__device__ __forceinline__ uint32_t gelu_h2(float lo, float hi) {
  const __half2 x = h2_pack_sat(lo, hi);
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.0f));
  const __half2 p = __hfma2(x2, __float2half2_rn(WJ_GELU_C3), __float2half2_rn(WJ_GELU_C1));
  const __half2 t = h2_tanh_approx(__hmul2(x, p));
  const __half2 hp = __hfma2(t, __float2half2_rn(0.5f), __float2half2_rn(0.5f));
  return h2_to_bf16x2(__hmul2(x, hp));
}
__device__ __forceinline__ void gelu_h2_save(float lo, float hi, uint32_t& g, uint32_t& dg) {
  const __half2 x = h2_pack_sat(lo, hi);
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.0f));
  const __half2 p = __hfma2(x2, __float2half2_rn(WJ_GELU_C3), __float2half2_rn(WJ_GELU_C1));
  const __half2 t = h2_tanh_approx(__hmul2(x, p));
  const __half2 hp = __hfma2(t, __float2half2_rn(0.5f), __float2half2_rn(0.5f));
  g = h2_to_bf16x2(__hmul2(x, hp));
  const __half2 q = __hfma2(x2, __float2half2_rn(3.0f * WJ_GELU_C3), __float2half2_rn(WJ_GELU_C1));
  const __half2 s = __hfma2(__hneg2(t), t, __float2half2_rn(1.0f));
  const __half2 r = __hmul2(__hmul2(x, s), q);
  dg = h2_to_bf16x2(__hfma2(r, __float2half2_rn(0.5f), hp));
}
// gelu'(lo), gelu'(hi) as fp32 (backward of the first conv block recomputes the factor instead of reading a saved copy)
__device__ __forceinline__ float2 dgelu_h2(float lo, float hi) {
  const __half2 x = h2_pack_sat(lo, hi);
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(100.0f));
  const __half2 p = __hfma2(x2, __float2half2_rn(WJ_GELU_C3), __float2half2_rn(WJ_GELU_C1));
  const __half2 t = h2_tanh_approx(__hmul2(x, p));
  const __half2 hp = __hfma2(t, __float2half2_rn(0.5f), __float2half2_rn(0.5f));
  const __half2 q = __hfma2(x2, __float2half2_rn(3.0f * WJ_GELU_C3), __float2half2_rn(WJ_GELU_C1));
  const __half2 s = __hfma2(__hneg2(t), t, __float2half2_rn(1.0f));
  const __half2 r = __hmul2(__hmul2(x, s), q);
  return __half22float2(__hfma2(r, __float2half2_rn(0.5f), hp));
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
// fp32 -> nearest tf32 (ties away from zero), kept as an fp32 word with the low 13 mantissa bits zero.  The tensor core
// truncates raw fp32 operands, which doubles the error of the TF32 inference path; operands are rounded as written.
__device__ __forceinline__ float tf32_round(float x) {
  uint32_t y;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(y) : "f"(x));
  return __uint_as_float(y);
}
// Two values rounded to bf16 (round-to-nearest-even) and widened again with ONE pack (F2FP) + two integer ops instead
// of two F2F conversions: F2F shares the quarter-rate XU pipe with MUFU, which the GELU epilogues saturate.
__device__ __forceinline__ void bf16_round2(float& a, float& b) {
  const uint32_t w = pack_bf16x2(a, b);
  a = __uint_as_float(w << 16);
  b = __uint_as_float(w & 0xffff0000u);
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace wj
