// sm_100a PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld),
// UMMA shared-memory + instruction descriptors, system-scope release/acquire for cross-GPU flags.
//
// Everything here is hand-written inline PTX for Blackwell (B200, compute_100a).  No CUTLASS/CuTe
// types are used; descriptor bit layouts follow the PTX ISA "tcgen05 matrix descriptor" /
// "instruction descriptor" tables.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sky {

// ----------------------------------------------------------------------------------------------
// misc
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 %%rx;\n"
      ".reg .pred %%px;\n"
      "elect.sync %%rx|%%px, %1;\n"
      "@%%px mov.s32 %0, 1;\n"
      "}\n"
      : "+r"(pred)
      : "r"(0xffffffffu));
  return pred != 0;
}

__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Programmatic dependent launch: wait until the previous grid in the stream has completed (and its
// memory is visible); allow the next grid to start launching.  No-ops without the launch attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
// 2D tiled load global -> shared, completion signalled on an mbarrier (complete_tx::bytes).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar,
                                            int c_inner, int c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4}], [%2];"
      ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer)
      : "memory");
}

// 3D tiled load (inner, middle, outer coordinates); out-of-range elements are zero-filled, which
// is how the tiled attention kernels read ragged last tiles of a sequence.
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// 4D tiled load; the tiled attention kernels for head sizes other than 64 (zero-filled columns
// past the head size as well as rows past the sequence end).
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar,
                                            int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// tcgen05.commit: arrive on an mbarrier once all previously issued MMAs of this thread completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// CTA pair (cta_group::2): two CTAs of a 2-cluster (same TPC) run ONE UMMA of M = 256.  Each CTA
// stages its own 128 rows of A and HALF of the B tile; the leader (cluster rank 0) issues the
// MMAs, which read both CTAs' shared memory and write both CTAs' TMEM.  This cuts the bytes each
// CTA pulls from L2 by a third; measured effect and when it pays: profiles/gemm_schedules.md.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n"
               "barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr)
               : "memory");
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
// distributed shared memory: store two floats into another CTA of the cluster
__device__ __forceinline__ void st_cluster_v2_f32(uint32_t cluster_addr, float a, float b) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(cluster_addr), "f"(a), "f"(b)
               : "memory");
}
// wait on a LOCAL mbarrier whose arrivals (and the data they publish) come from other CTAs of the
// cluster: acquire at cluster scope
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
// TMA load whose completion bytes land on a barrier that may live in the PEER CTA
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tmap,
                                                 uint32_t bar_cluster_addr, int c_inner,
                                                 int c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(bar_cluster_addr), "r"(c_inner), "r"(c_outer)
      : "memory");
}
// same, multicast: the box lands at the same CTA-relative offset in every CTA of `mask`; the
// completion bytes go to the barrier at `bar_addr`'s offset in each destination's pair leader
__device__ __forceinline__ void tma_load_2d_pair_mc(void* smem_dst, const CUtensorMap* tmap,
                                                    uint32_t bar_addr, int c_inner, int c_outer,
                                                    uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      ".multicast::cluster [%0], [%1, {%4, %5}], [%2], %3;"
      ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(bar_addr), "h"(mask), "r"(c_inner), "r"(c_outer)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// commit: arrive on the barrier at this offset in BOTH CTAs of the pair once the MMAs retired
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(mask)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a,
                                                  uint64_t desc_b, uint32_t idesc,
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

// ----------------------------------------------------------------------------------------------
// tcgen05: descriptors
// ----------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_128B.  Bit layout (PTX ISA):
//   [0,14)  start address >> 4      [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4     [46,48) version (1 on sm_100)
//   [49,52) base offset (0: tiles are 1024B aligned)   [61,64) swizzle mode (2 = 128B)
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                         uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// Instruction descriptor for kind::f16 with BF16 A/B and FP32 accumulate.
//   [4,6) D format (1 = f32)   [7,10) A format (1 = bf16)   [10,13) B format (1 = bf16)
//   [15]  A major (0 = K, 1 = MN)   [16] B major   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_bf16_f32(int umma_m, int umma_n, bool a_mn,
                                                           bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn) << 15) |
         (static_cast<uint32_t>(b_mn) << 16) | (static_cast<uint32_t>(umma_n >> 3) << 17) |
         (static_cast<uint32_t>(umma_m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by a single thread.
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05: TMEM -> registers (32 lanes x 32 columns of 32-bit per warp)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
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
// registers -> TMEM (same 32 lanes x 32 columns shape): lets an epilogue park a transformed tile
// in the accumulator's own columns between two passes (GEMM + LayerNorm epilogue)
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]),
        "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]),
        "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
        "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
        "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// cross-GPU flags (system scope)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void red_release_sys_add(uint32_t* addr, uint32_t v) {
  asm volatile("red.release.sys.global.add.u32 [%0], %1;" ::"l"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* addr) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* addr) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(addr) : "memory");
  return v;
}
// Spin until *addr >= target (monotonic counters). Returns false on timeout (ns budget).
__device__ __forceinline__ bool wait_flag_ge(const uint32_t* addr, uint32_t target,
                                             uint64_t timeout_ns) {
  if (ld_acquire_sys(addr) >= target) return true;
  const uint64_t t0 = globaltimer_ns();
  while (true) {
    if (ld_acquire_sys(addr) >= target) return true;
    if (globaltimer_ns() - t0 > timeout_ns) return false;
    __nanosleep(64);
  }
}

// ----------------------------------------------------------------------------------------------
// small math helpers shared by epilogues
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(h);
}

// erf-form GELU as used by BERT (x * 0.5 * (1 + erf(x / sqrt(2)))).
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f));
}
// d/dx gelu_erf(x) = Phi(x) + x * phi(x)
__device__ __forceinline__ float dgelu_erf(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

// Fast variants for GEMM epilogues (Abramowitz-Stegun 7.1.26 erf, |err| < 1.5e-7 - far below
// bf16 resolution): one MUFU.RCP + one MUFU.EX2 + 6 FMA instead of libdevice erff.
__device__ __forceinline__ float erf_exp_fast(float z_abs, float& e_out) {
  // returns erf(z_abs) for z_abs >= 0 and e_out = exp(-z^2)
  // rcp.approx (one MUFU): __frcp_rn expands to MUFU + Newton steps + a slow-path branch per
  // element, which serialised the whole epilogue (tools/triage_gemm.py: +30 us on FFN1)
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z_abs, 1.0f)));
  float poly = 1.061405429f;
  poly = fmaf(poly, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  poly *= t;
  e_out = __expf(-z_abs * z_abs);
  return fmaf(-poly, e_out, 1.0f);
}
__device__ __forceinline__ float gelu_fast(float x) {
  float e;
  const float er = erf_exp_fast(fabsf(x) * 0.70710678118654752f, e);
  return 0.5f * x * (1.0f + copysignf(er, x));
}
__device__ __forceinline__ float dgelu_fast(float x) {
  float e;  // exp(-x^2/2)
  const float er = erf_exp_fast(fabsf(x) * 0.70710678118654752f, e);
  const float cdf = 0.5f * (1.0f + copysignf(er, x));
  return fmaf(x * 0.3989422804014327f, e, cdf);
}
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void red_add_v4_f32(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c),
               "f"(d)
               : "memory");
}

// Counter-based RNG for dropout: splitmix64 of (seed, element-group index) -> 4 x 16-bit lanes.
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// Effective per-step seed: {seed, step} live in device memory so CUDA-graph replays advance it.
__device__ __forceinline__ uint64_t dropout_seed(const uint64_t* rng_state, uint32_t stream) {
  return splitmix64(rng_state[0] + 0x632BE59BD9B4E019ull * (rng_state[1] + 1)) ^
         (static_cast<uint64_t>(stream) << 32);
}
// keep-mask for 4 consecutive elements starting at element index `idx4*4`; thr16 = p * 65536.
__device__ __forceinline__ uint32_t dropout_keep4(uint64_t seed, uint64_t idx4, uint32_t thr16) {
  const uint64_t r = splitmix64(seed ^ (idx4 * 0xD1342543DE82EF95ull));
  uint32_t m = 0;
  m |= (static_cast<uint32_t>(r & 0xFFFF) >= thr16) ? 1u : 0u;
  m |= (static_cast<uint32_t>((r >> 16) & 0xFFFF) >= thr16) ? 2u : 0u;
  m |= (static_cast<uint32_t>((r >> 32) & 0xFFFF) >= thr16) ? 4u : 0u;
  m |= (static_cast<uint32_t>((r >> 48) & 0xFFFF) >= thr16) ? 8u : 0u;
  return m;
}

}  // namespace sky
